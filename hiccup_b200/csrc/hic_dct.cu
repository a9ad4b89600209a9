// hic_dct.cu -- DCT-mode transform stage: K1 (fused colour + pyrDown + DCT + quantise + zigzag),
// the float64 tie fix-up, K7 (dequantise + IDCT) and K8 (pyrUp + colour), their thumbnail, region and scaled
// variants, plus layout converters.
//
// Data layout in HBM (see include/hiccup_b200.h): RGB u8 interleaved in; coefficients as int16
// "zigzag blocks" (one 128-byte line per 8x8 block) out.  HBM-bound by design: 3 B/pixel read,
// 3 B/pixel written (1.5 samples/pixel x 2 B) = 6 algorithmic bytes per pixel for K1.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <type_traits>
#include "hic_core.cuh"
#include "hic_dct_bound.h"
#include "hic_f32x2.cuh"
#include "hic_runtime.cuh"

namespace hic {

// ------------------------------------------------------------------------------------------------
// constant tables (per device)
// ------------------------------------------------------------------------------------------------
struct DctTables {
    float2 rq2[2][64];   // [0 = luminance, 1 = chroma][natural index]: 4 / (scale_u scale_v q), twice (both f32x2 lanes)
    float rq[2][64];     // the same once (the one-block-per-thread variant pairs neighbouring columns)
    float kq[2][64];     // near-tie band per unit E: kappa(u, v) * margin * 4 u / q   (0 for DC: it is exact)
    float dq[2][64];     // q prescale_u prescale_v / 256 (inverse)
    float qw[2][64];     // inverse band weight: q * w(u, v) * margin
    int qi[2][64];       // q
    int izz[64];         // natural index -> scan position
    float sqw[2][2][16]; // scaled decode band weight [0: M = 4, 1: M = 2][kind][M u + v]: T(u, v) * w_s(u, v) * margin
};
__constant__ DctTables c_tab;
__constant__ uint8_t c_zigzag[64] = HIC_ZIGZAG8;

static const int h_lum[64] = HIC_LUM_TABLE;
static const int h_chroma[64] = HIC_CHROMA_TABLE;
static const uint8_t h_zigzag[64] = HIC_ZIGZAG8;

static int ensure_tables() {
    static std::mutex mu;
    static bool done[64] = {false};
    int dev = 0;
    HIC_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev < 64 && done[dev]) return HIC_OK;
    static DctTables t;
    static bool built = false;
    if (!built) {
        const DctBounds bounds = dct_bounds();          // rigorous float32 error bounds of the transforms (hic_dct_bound.h)
        const double u24 = 1.0 / 16777216.0;
        for (int kind = 0; kind < 2; ++kind)
            for (int u = 0; u < 8; ++u)
                for (int v = 0; v < 8; ++v) {
                    const int nat = 8 * u + v;
                    const int q = (kind == 0 ? h_lum : h_chroma)[nat];
                    const float rq = (float)(4.0 / (eo_forward_scale(u) * eo_forward_scale(v) * q));
                    t.rq2[kind][nat] = make_float2(rq, rq);
                    t.rq[kind][nat] = rq;
                    t.kq[kind][nat] = nat == 0 ? 0.f : (float)(bounds.kappa_fwd[nat] * HIC_BAND_MARGIN * 4.0 * u24 / q);
                    t.dq[kind][nat] = (float)(q * eo_inverse_prescale(u) * eo_inverse_prescale(v) / 256.0);
                    t.qw[kind][nat] = (float)(q * bounds.w_inv[nat] * HIC_BAND_MARGIN);
                    t.qi[kind][nat] = q;
                }
        for (int k = 0; k < 64; ++k) t.izz[h_zigzag[k]] = k;
        double w4[16], w2[4];
        scaled_bounds<4>(w4);
        scaled_bounds<2>(w2);
        for (int kind = 0; kind < 2; ++kind)
            for (int u = 0; u < 4; ++u)
                for (int v = 0; v < 4; ++v) {
                    const int q = (kind == 0 ? h_lum : h_chroma)[8 * u + v];
                    t.sqw[0][kind][4 * u + v] = (float)(q * w4[4 * u + v] * HIC_BAND_MARGIN);
                    if (u < 2 && v < 2) t.sqw[1][kind][2 * u + v] = (float)(q * w2[2 * u + v] * HIC_BAND_MARGIN);
                }
        built = true;
    }
    HIC_CUDA(cudaMemcpyToSymbol(c_tab, &t, sizeof(t)));
    if (dev < 64) done[dev] = true;
    return HIC_OK;
}

// ------------------------------------------------------------------------------------------------
// geometry
// ------------------------------------------------------------------------------------------------
static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

static int geometry_of(int h, int w, hic_dct_geometry* g) {
    HIC_REQUIRE(g != nullptr, "geometry output is NULL");
    HIC_REQUIRE(h >= 2 && w >= 2, "image must be at least 2x2 (got %dx%d)", h, w);
    HIC_REQUIRE(h <= 65536 && w <= 65536, "image larger than 65536 on a side (got %dx%d)", h, w);
    g->h = h;
    g->w = w;
    g->hc = h / 2;
    g->wc = w / 2;
    g->nby_l = ceil_div(h, 8);
    g->nbx_l = ceil_div(w, 8);
    g->nby_c = ceil_div(g->hc, 8);
    g->nbx_c = ceil_div(g->wc, 8);
    g->nb_l = (int64_t)g->nby_l * g->nbx_l;
    g->nb_c = (int64_t)g->nby_c * g->nbx_c;
    g->blocks_per_image = g->nb_l + 2 * g->nb_c;
    g->out_h = 2 * g->hc;
    g->out_w = 2 * g->wc;
    return HIC_OK;
}

// ------------------------------------------------------------------------------------------------
// region decode: the blocks a window of the output reads
// ------------------------------------------------------------------------------------------------
// Output pixel (oy, ox) reads luminance sample (oy, ox) and K8's chroma taps: rows cy - 1 .. cy + 1 of cy = oy / 2
// (row 1 for cy = 0, clamped to hc - 1 at the bottom), the same for columns.  So a window of rh output rows at top
// reads luminance rows [top, top + rh - 1] and chroma rows [max(0, top/2 - 1), min(hc - 1, (top + rh - 1)/2 + 1)]
// -- at most rh / 2 + 3 of them.  Every window of one size gets a block rectangle of one size per plane kind: the
// most blocks those rows (columns) can touch, at most the plane's block count.  It starts at the block of the first
// row the window reads, moved back where it would run past the plane's last block.
// The scaled region decode uses the same rules at M = 8 / scale samples per block side: a window of the 1/scale image
// reads rows of the reduced planes (M nby_l x M nbx_l luminance, M nby_c x M nbx_c chroma) exactly as a window of the
// full decode reads rows of the full-size planes, so only the block size changes.
struct RegionSpan {
    int ny_l, nx_l;   // luminance rectangle, blocks
    int ny_c, nx_c;   // chroma rectangle (Cr and Cb alike)
};

template <int M>
constexpr int log2_side() { return M == 8 ? 3 : (M == 4 ? 2 : 1); }
template <int M>
__host__ __device__ inline int region_span_l(int r, int nb) { return min(nb, (r + M - 2) / M + 1); }   // r samples
template <int M>
__host__ __device__ inline int region_span_c(int r, int nb) { return min(nb, (r / 2 + 3 + M - 2) / M + 1); }
template <int M>
__host__ __device__ inline RegionSpan region_span(const hic_dct_geometry& g, int rh, int rw) {
    return {region_span_l<M>(rh, g.nby_l), region_span_l<M>(rw, g.nbx_l), region_span_c<M>(rh, g.nby_c), region_span_c<M>(rw, g.nbx_c)};
}
// first block row (column) of the luminance / chroma rectangle of a window whose first output row (column) is t
template <int M>
__host__ __device__ inline int region_first_l(int t, int span, int nb) { return min(t >> log2_side<M>(), nb - span); }
template <int M>
__host__ __device__ inline int region_first_c(int t, int span, int nb) {
    return min(max(0, (t >> 1) - 1) >> log2_side<M>(), nb - span);
}

// a window of the decoded image (scale 1) or of its 1/scale image, ceil(out_h / scale) x ceil(out_w / scale)
static int region_check(const hic_dct_geometry& g, int64_t top, int64_t left, int64_t rh, int64_t rw, int scale = 1) {
    HIC_REQUIRE(rh >= 1 && rw >= 1, "empty region %lldx%lld", (long long)rh, (long long)rw);
    const int ih = (g.out_h + scale - 1) / scale, iw = (g.out_w + scale - 1) / scale;
    const bool inside = top >= 0 && left >= 0 && top + rh <= ih && left + rw <= iw;
    if (scale == 1)
        HIC_REQUIRE(inside, "region %lldx%lld at (%lld, %lld) is not inside the %dx%d decoded image", (long long)rh,
                    (long long)rw, (long long)top, (long long)left, ih, iw);
    HIC_REQUIRE(inside, "region %lldx%lld at (%lld, %lld) is not inside the %dx%d 1/%d-scale image", (long long)rh,
                (long long)rw, (long long)top, (long long)left, ih, iw, scale);
    return HIC_OK;
}

// {by, bx, nby, nbx} of the luminance rectangle, then of each chroma rectangle, of a window at (top, left)
template <int M>
static void region_rect(const hic_dct_geometry& g, int top, int left, int rh, int rw, int32_t* rect) {
    const RegionSpan s = region_span<M>(g, rh, rw);
    const int32_t out[8] = {region_first_l<M>(top, s.ny_l, g.nby_l), region_first_l<M>(left, s.nx_l, g.nbx_l), s.ny_l, s.nx_l,
                            region_first_c<M>(top, s.ny_c, g.nby_c), region_first_c<M>(left, s.nx_c, g.nbx_c), s.ny_c, s.nx_c};
    memcpy(rect, out, sizeof(out));
}

// window-local tiles of one image (bytes, M x M samples per block) and the work buffer: n origins, then the n images'
// Y tiles, Cr tiles, Cb tiles
struct RegionLayout {
    RegionSpan s;
    size_t head, ly, lc, total;
    uint64_t blocks;      // selected blocks of the batch
};
template <int M>
static RegionLayout region_layout(int n, const hic_dct_geometry& g, int rh, int rw) {
    RegionLayout L;
    L.s = region_span<M>(g, rh, rw);
    L.head = ((size_t)n * 2 * sizeof(int32_t) + 255) / 256 * 256;
    L.ly = (size_t)M * M * L.s.ny_l * L.s.nx_l;
    L.lc = (size_t)M * M * L.s.ny_c * L.s.nx_c;
    L.total = L.head + (size_t)n * (L.ly + 2 * L.lc);
    L.blocks = (uint64_t)n * (L.ly + 2 * L.lc) / (M * M);
    return L;
}

// ------------------------------------------------------------------------------------------------
// K1: fused encode transform
// ------------------------------------------------------------------------------------------------
namespace k1 {
// Tile: 128 x 64 luminance pixels = 16 x 8 Y blocks + 8 x 4 Cr blocks + 8 x 4 Cb blocks = 192 blocks.
// In the transform stage a thread carries one block, two rows (then two columns) in each packed f32x2
// register pair -- 192 threads per tile.  The quantised blocks are staged in shared memory (the RGB region
// is dead by then) in the 128-byte-swizzle pattern and leave through two TMA tensor stores: a thread's
// eight 16-byte pieces of its 128-byte block would otherwise be a global store of 32 different lines per
// warp instruction, and those stores alone were half of the kernel's LSU wavefronts.
// The staged RGB region covers image columns x0-16 .. x0+132 and rows y0-2 .. y0+64 (pyrDown needs
// columns x0-2 .. x0+128 and rows y0-2 .. y0+64).  The 16-pixel lead is what TMA demands: the innermost
// start offset of a box must be a multiple of 16 bytes (a 12-byte-aligned start faults with "illegal
// instruction"; probed in tools/scratch/tma_test.cu), and 3 * (x0 - lead) is a multiple of 16 only for
// lead = 0 mod 16.
#ifndef HIC_K1_TH
#define HIC_K1_TH 64
#endif
#ifndef HIC_K1_PF_WAVES
#define HIC_K1_PF_WAVES 2          // L2 prefetch distance in waves of resident CTAs (0: none)
#endif
constexpr int TW = 128;
constexpr int TH = HIC_K1_TH;          // tile height: 64 (4 CTAs per SM) or 32 (7 lighter CTAs per SM)
constexpr int CTAS_PER_SM = TH == 64 ? 4 : 7;
constexpr int RH = TH + 3;            // staged rows
constexpr int RWORDS = 112;           // staged row pitch in 32-bit words (448 bytes = 149 pixels)
constexpr int RPIX = 136;             // pixels converted per staged row (34 groups of 4)
constexpr int RGROUPS = RPIX / 4;
constexpr int LEAD = 16;              // staged pixel q <-> image column x0 - LEAD + q
constexpr int SKIP = 12;              // converted pixel p = q - SKIP <-> image column x0 - 4 + p
constexpr int SPIX = RWORDS * 4 / 3;  // whole pixels in a staged row
constexpr int C_PITCH = 136;          // Cr/Cb staging pitch (bytes), indexed by region pixel (34 groups of 4)
constexpr int CW = TW / 2;            // chroma tile
constexpr int CH = TH / 2;
constexpr int CD_PITCH = CW + 8;      // pitch of the downsampled chroma tiles: block rows land in different banks
constexpr int NY_BLOCKS = (TW / 8) * (TH / 8);       // 128
constexpr int NC_BLOCKS = (CW / 8) * (CH / 8);       // 32 per chroma plane
constexpr int THREADS = NY_BLOCKS + 2 * NC_BLOCKS;   // one block per thread: 192
constexpr int WARPS = THREADS / 32;
constexpr float MAGIC = 12582912.0f;                 // 1.5 * 2^23: float add rounds to integer, RN-even
// The staged region can arrive as LOAD_CHUNKS TMA boxes of CHUNK_ROWS rows, each with its own barrier, so that stage 1
// starts on the first rows while the rest is in flight.  Measured on C2: two boxes 0.566 ms against 0.543 ms for one
// (the second wait and the second descriptor cost more than the earlier start gains; four boxes of 18 rows do not fit
// the shared-memory budget of four CTAs per SM) -- so one box it is.
constexpr int LOAD_CHUNKS = 1;
constexpr int CHUNK_ROWS = 2 * ((RH + 2 * LOAD_CHUNKS - 1) / (2 * LOAD_CHUNKS));
constexpr uint32_t CHUNK_BYTES = CHUNK_ROWS * RWORDS * 4;
static_assert(CHUNK_BYTES % 128 == 0, "a TMA box lands on a 128-byte boundary of shared memory (an even number of 448-byte rows)");

// Colour conversion constants (cv2's 14-bit fixed point, compression.py:21), scaled by 4 so that every
// result lands in byte 2 of its accumulator and the packing PRMTs pick it up without a shift:
//   Y  = (4899 R + 9617 G + 1868 B + 8192) >> 14                 = byte 2 of two 16x8-bit dot products
//   Cr = ((R - Y) 11682 + (128 << 14) + 8192) >> 14, clamped     = byte 2 of min(46728 R - 46728 Y + C4, 2^24 - 1)
//   Cb = ((B - Y)  9241 + (128 << 14) + 8192) >> 14              = byte 2 of      36964 B - 36964 Y + C4
// R - Y spans [-179, 179] and B - Y [-226, 226] (extremes of cv2's weights): Cr reaches 256 only at the
// top (hence the min) and never goes below 0; Cb stays inside 1..255.  All arithmetic instead of the
// shared-memory lookup tables of the first version: the kernel's stalls were on the shared-memory pipe.
constexpr uint32_t W_RG = (4u * 9617u << 16) | (4u * 4899u);     // dp2a.lo: R (byte 0) and G (byte 1)
constexpr uint32_t W_B = 4u * 1868u;                             // dp2a.hi: B (byte 2); byte 3 weighs 0
constexpr uint32_t K_CR = 4u * 11682u, K_CB = 4u * 9241u;
constexpr uint32_t C4 = 4u * ((128u << 14) + 8192u);
struct Smem {
    union alignas(1024) {
        uint32_t rgb[LOAD_CHUNKS * CHUNK_ROWS * RWORDS];      // stage 0/1 (TMA destination)
        uint16_t hpass[2][RH][CW];                   // stage 2 (rgb is dead by then)
        int4 stage[THREADS * 8];                     // stage 3 -> TMA stores (hpass is dead by then): block t = row t, 128-byte swizzle
    };
    alignas(16) uint8_t y[TH][TW];
    union alignas(16) {
        uint8_t cr[RH][C_PITCH];                     // stage 1 -> 2a
        uint8_t crd[CH][CD_PITCH];                   // stage 2b -> 3 (cr is dead by then)
    };
    union alignas(16) {
        uint8_t cb[RH][C_PITCH];
        uint8_t cbd[CH][CD_PITCH];
    };
    alignas(8) unsigned long long bar[LOAD_CHUNKS];
};
static_assert(sizeof(Smem) <= (TH == 64 ? 57344 : 32256), "CTAS_PER_SM CTAs per SM: (228 KB - 1 KB reserved each) / CTAS_PER_SM");
static_assert(sizeof(int4) * THREADS * 8 <= sizeof(uint32_t) * RH * RWORDS, "the staged blocks fit in the RGB region");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One 8x8 block per thread: the row pass in scalar float32, the column pass and the quantiser packed (two columns
// per f32x2 register).  The quantised zigzag int16 of the block go to its 128-byte row of the
// staging area, 16-byte piece j at position j ^ sw (the TMA 128-byte swizzle; sw = row & 7), so that the
// eight threads of a quarter warp hit all 32 banks.  rows / cols < 8: the block hangs over the bottom /
// right edge of its plane -- the reference crops the coefficient plane back to the channel shape
// (transform.py:63) and re-pads it with zeros (codec.py:288,294), so coefficients at vertical frequency
// >= rows or horizontal frequency >= cols are zero.
__device__ __forceinline__ unsigned transform_single(int kind, const uint32_t (&wv)[16], int4* __restrict__ out, int sw,
                                                     int rows, int cols) {
    uint32_t abs_sum = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) abs_sum = __vsadu4(wv[i], 0x80808080u) + abs_sum;
    const float fe = (float)abs_sum;
    // Row pass in scalar float32, one row at a time; column pass packed, two columns per f32x2 register.  (Both
    // passes packed -- two rows, then two columns per register -- needs the 64 values re-paired in between, and the
    // register moves of that re-pairing were nearly as many as the packed operations they served: 0.557 ms against
    // 0.549 ms on C2.  Same operations per value, same roundings: the results are bit-identical.)
    const float shift = -(8388608.0f + 128.0f);
    float T[64];     // T[r * 8 + v] = row-transformed row r, horizontal frequency v
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        float x[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) x[c] = __uint_as_float(__byte_perm(wv[2 * r + (c >> 2)], 0x4B000000u, 0x7540 + (c & 3)));
        float s[4], d[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            d[i] = x[i] - x[7 - i];
            s[i] = fmaf(2.0f, x[7 - i] + shift, d[i]);
        }
        eo_forward8_tail(s[0], s[1], s[2], s[3], d[0], d[1], d[2], d[3], T[8 * r + 0], T[8 * r + 1], T[8 * r + 2],
                         T[8 * r + 3], T[8 * r + 4], T[8 * r + 5], T[8 * r + 6], T[8 * r + 7]);
    }
    f2 b[32];        // b[u * 4 + cp] = coefficients (u, 2 cp) and (u, 2 cp + 1)
#pragma unroll
    for (int cp = 0; cp < 4; ++cp) {
        f2 d[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) d[r] = f2(T[8 * r + 2 * cp], T[8 * r + 2 * cp + 1]);
        eo_forward8(d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7]);
#pragma unroll
        for (int r = 0; r < 8; ++r) b[r * 4 + cp] = d[r];
    }
    float worst = 0.f;
    const f2 magic2(MAGIC);
    const float* __restrict__ rqt = c_tab.rq[kind];
    const float* __restrict__ kqt = c_tab.kq[kind];
#pragma unroll
    for (int p = 0; p < 32; ++p) {
        const int n0 = (p >> 2) * 8 + 2 * (p & 3);
        f2 rq;
        rq.v = *reinterpret_cast<const unsigned long long*>(&rqt[n0]);
        const f2 t = fma2(b[p], rq, magic2);
        const f2 d = fma2(b[p], rq, magic2 - t);
        b[p] = t;
        if (p != 0) worst = fmaxf(worst, fmaf(fe, kqt[n0], fabsf(d.lo())));      // DC is exact
        worst = fmaxf(worst, fmaf(fe, kqt[n0 + 1], fabsf(d.hi())));
    }
    if (rows < 8 || cols < 8) {          // (edge blocks of shapes that are not multiples of 8: MAGIC carries a zero)
#pragma unroll
        for (int p = 0; p < 32; ++p) {
            const int u = p >> 2, v0 = 2 * (p & 3);
            const float lo = (u >= rows || v0 >= cols) ? MAGIC : b[p].lo();
            const float hi = (u >= rows || v0 + 1 >= cols) ? MAGIC : b[p].hi();
            b[p] = f2(lo, hi);
        }
    }
    constexpr uint8_t zz[64] = HIC_ZIGZAG8;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        int4 w4;
        int* pw = reinterpret_cast<int*>(&w4);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int n_lo = zz[8 * j + 2 * e], n_hi = zz[8 * j + 2 * e + 1];
            const f2 t0 = b[(n_lo >> 3) * 4 + ((n_lo & 7) >> 1)], t1 = b[(n_hi >> 3) * 4 + ((n_hi & 7) >> 1)];
            const int v0 = __float_as_int((n_lo & 1) ? t0.hi() : t0.lo()), v1 = __float_as_int((n_hi & 1) ? t1.hi() : t1.lo());
            pw[e] = __byte_perm(v0, v1, 0x5410);
        }
        out[j ^ sw] = w4;
    }
    return worst >= 0.499999f ? 1u : 0u;
}

// Which block thread `tid` of tile (tbx, tby) of image `img` carries: threads 0..NY_BLOCKS-1 the luminance
// blocks of the tile row by row, then the Cr and the Cb blocks.  false: the block lies outside its plane.
struct TileBlock {
    uint32_t index;        // block index in the coefficient buffer
    int kind;              // 0 = luminance, 1 = chroma
    int by, bx;            // block position inside the tile
    int plane;             // 0 = Cr, 1 = Cb (chroma)
    int rows, cols;        // samples of the block inside its plane (>= 8: all)
};
__device__ __forceinline__ bool tile_block(int tid, int tbx, int tby, int img, const hic_dct_geometry& g, int h, int w,
                                           TileBlock& t) {
    if (tid < NY_BLOCKS) {
        t.kind = 0;
        t.plane = 0;
        t.by = tid / (TW / 8);
        t.bx = tid % (TW / 8);
        const int BY = tby * (TH / 8) + t.by, BX = tbx * (TW / 8) + t.bx;
        t.index = (uint32_t)((int64_t)img * g.blocks_per_image + (int64_t)BY * g.nbx_l + BX);
        t.rows = h - 8 * BY;
        t.cols = w - 8 * BX;
        return BY < g.nby_l && BX < g.nbx_l;
    }
    t.kind = 1;
    t.plane = (tid - NY_BLOCKS) / NC_BLOCKS;
    const int local = (tid - NY_BLOCKS) % NC_BLOCKS;
    t.by = local / (CW / 8);
    t.bx = local % (CW / 8);
    const int BY = tby * (CH / 8) + t.by, BX = tbx * (CW / 8) + t.bx;
    t.index = (uint32_t)((int64_t)img * g.blocks_per_image + g.nb_l + (int64_t)t.plane * g.nb_c + (int64_t)BY * g.nbx_c + BX);
    t.rows = g.hc - 8 * BY;
    t.cols = g.wc - 8 * BX;
    return BY < g.nby_c && BX < g.nbx_c;
}

// K1 leaves one word per warp: the ballot of its threads' near-tie flags (a plain store -- a slot request
// through an atomic made every warp wait for the round trip at the end of its tile).  This kernel turns the
// words into the list of flagged blocks the fix-up kernel works through.
__global__ void __launch_bounds__(256)
tie_list_kernel(const uint32_t* __restrict__ flagmap, uint32_t n_words, int tiles_x, int tiles_y, hic_dct_geometry g, int h,
                int w, hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    const unsigned lane = threadIdx.x & 31;
    for (uint32_t base = (blockIdx.x * blockDim.x + threadIdx.x) - lane; base < n_words; base += gridDim.x * blockDim.x) {
        const uint32_t wi = base + lane;
        const uint32_t m = wi < n_words ? flagmap[wi] : 0u;
        const uint32_t cnt = __popc(m);
        uint32_t incl = cnt;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= (unsigned)off) incl += o;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) continue;
        uint32_t slot = 0;
        if (lane == 0) slot = atomicAdd(&stats[0], total);
        slot = __shfl_sync(0xffffffffu, slot, 0) + incl - cnt;
        const uint32_t tile = wi / WARPS, warp = wi - tile * WARPS;
        const int tbx = (int)(tile % tiles_x), tby = (int)((tile / tiles_x) % tiles_y), img = (int)(tile / ((uint32_t)tiles_x * tiles_y));
        for (uint32_t rest = m; rest; rest &= rest - 1, ++slot) {
            TileBlock t;
            tile_block((int)(warp * 32 + __ffs(rest) - 1), tbx, tby, img, g, h, w, t);
            if (slot < tie_capacity) {
                hic_tie_record rec;
                rec.block = t.index;
                rec.reserved = 0;
                rec.mask = ~0ull;
                ties[slot] = rec;
            } else {
                atomicAdd(&stats[3], 1u);
            }
        }
    }
}

// tmap: the RGB batch with a whole tile as its box (L2 prefetch), tmap_rows: with a CHUNK_ROWS-row box (loads); tmap_l / tmap_c: the luminance / chroma blocks of the coefficient buffer (stores).
template <bool USE_TMA>
__global__ void __launch_bounds__(THREADS, CTAS_PER_SM)
forward_kernel(const __grid_constant__ CUtensorMap tmap, const __grid_constant__ CUtensorMap tmap_rows, const __grid_constant__ CUtensorMap tmap_l,
               const __grid_constant__ CUtensorMap tmap_c, const uint8_t* __restrict__ rgb, int h, int w,
               hic_dct_geometry g, uint32_t* __restrict__ flagmap) {
    constexpr int R16 = THREADS / 16;          // rows per step of the 16-lanes-per-row stages
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    Smem& s = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x;
    const int img = blockIdx.z;
    const int x0 = blockIdx.x * TW, y0 = blockIdx.y * TH;

    // ---- stage 0: RGB region -> shared memory ----
    if (USE_TMA) {
        if (tid == 0) {
#pragma unroll
            for (int c = 0; c < LOAD_CHUNKS; ++c) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&s.bar[c])));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            const int c0 = (3 * x0 - 3 * LEAD) / 4, c2 = img;
#pragma unroll
            for (int c = 0; c < LOAD_CHUNKS; ++c) {
                const uint32_t bar = smem_u32(&s.bar[c]);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(CHUNK_BYTES) : "memory");
                asm volatile(
                    "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                    ::"r"(smem_u32(s.rgb + c * CHUNK_ROWS * RWORDS)), "l"(reinterpret_cast<uint64_t>(&tmap_rows)), "r"(c0),
                    "r"(y0 - 2 + c * CHUNK_ROWS), "r"(c2), "r"(bar)
                    : "memory");
            }
            // pull the tile of a CTA two waves ahead (4 CTAs on each of 148 SMs per wave) into L2, so that
            // its own load finds the data there
            const unsigned per_img = gridDim.x * gridDim.y;
            const unsigned ahead = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x + (unsigned)HIC_K1_PF_WAVES * (unsigned)CTAS_PER_SM * 148u;
            if (HIC_K1_PF_WAVES > 0 && ahead < per_img * gridDim.z) {
                const unsigned pz = ahead / per_img, rem = ahead - pz * per_img;
                const unsigned py = rem / gridDim.x, pxb = rem - py * gridDim.x;
                const int p0 = (3 * (int)(pxb * TW) - 3 * LEAD) / 4, p1 = (int)(py * TH) - 2, p2 = (int)pz;
                asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global [%0, {%1, %2, %3}];"
                             ::"l"(reinterpret_cast<uint64_t>(&tmap)), "r"(p0), "r"(p1), "r"(p2) : "memory");
            }
        }
    }
    if (!USE_TMA) {
        // generic loader (row pitch not a multiple of 16 bytes): bytes with the border rule applied
        const uint8_t* src = rgb + (size_t)img * h * w * 3;
        uint8_t* dst8 = reinterpret_cast<uint8_t*>(s.rgb);
        for (int i = tid; i < RH * RPIX; i += THREADS) {
            const int ry = i / RPIX, p = SKIP + (i - ry * RPIX);
            const int gy = reflect101(y0 - 2 + ry, h), gx = reflect101(x0 - LEAD + p, w);
            const uint8_t* q = src + ((size_t)gy * w + gx) * 3;
            uint8_t* o = dst8 + ry * (RWORDS * 4) + p * 3;
            o[0] = q[0];
            o[1] = q[1];
            o[2] = q[2];
        }
    }
    __syncthreads();           // barriers initialised / generic load visible
    unsigned arrived = USE_TMA ? 0u : ~0u;             // chunks this thread has already seen complete
    auto wait_chunk = [&](int c) {
        if (!((arrived >> c) & 1u)) {
            asm volatile(
                "{\n"
                ".reg .pred P1;\n"
                "LAB_WAIT:\n"
                "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n"
                "@P1 bra DONE;\n"
                "bra LAB_WAIT;\n"
                "DONE:\n"
                "}\n" ::"r"(smem_u32(&s.bar[c]))
                : "memory");
            arrived |= 1u << c;
        }
    };
    if (USE_TMA) {
        // TMA zero-fills outside the image; cv2.pyrDown wants BORDER_REFLECT_101 there.  Only the
        // two pixels next to each edge are ever read by a valid output: patch them in place (edge tiles
        // wait for their whole region first).
        uint8_t* r8 = reinterpret_cast<uint8_t*>(s.rgb);
        const bool left = x0 == 0, right = x0 - LEAD + SPIX > w, top = y0 == 0, bottom = y0 - 2 + RH > h;
        if (left | right | top | bottom) {
#pragma unroll
            for (int c = 0; c < LOAD_CHUNKS; ++c) wait_chunk(c);
        }
        if (left | right) {
            for (int i = tid; i < RH * 4; i += THREADS) {
                const int ry = i >> 2, k = i & 3;
                // k = 0, 1: image columns -2, -1; k = 2, 3: image columns w, w + 1
                const int col = k < 2 ? k - 2 : w + (k - 2);
                if ((k < 2 && !left) || (k >= 2 && !right)) continue;
                const int p = col - x0 + LEAD, ps = reflect101(col, w) - x0 + LEAD;
                if (p < 0 || p >= SPIX || ps < 0 || ps >= SPIX) continue;
                uint8_t* o = r8 + ry * (RWORDS * 4);
                o[3 * p] = o[3 * ps];
                o[3 * p + 1] = o[3 * ps + 1];
                o[3 * p + 2] = o[3 * ps + 2];
            }
            __syncthreads();
        }
        if (top | bottom) {
            for (int i = tid; i < 4 * RWORDS; i += THREADS) {
                const int k = i / RWORDS, wd = i - k * RWORDS;
                const int row = k < 2 ? k - 2 : h + (k - 2);
                if ((k < 2 && !top) || (k >= 2 && !bottom)) continue;
                const int ry = row - y0 + 2, rs = reflect101(row, h) - y0 + 2;
                if (ry < 0 || ry >= RH || rs < 0 || rs >= RH) continue;
                s.rgb[ry * RWORDS + wd] = s.rgb[rs * RWORDS + wd];
            }
            __syncthreads();
        }
    }

    // ---- stage 1: colour conversion, four pixels (three words) at a time ----
    // Y = (4899 R + 9617 G + 1868 B + 8192) >> 14 as two dot products on the weight bytes.  Groups 1..32
    // of a row (the 128 tile columns) go one per lane, rows warp + WARPS k; the two halo groups per row
    // (columns x0-4..x0-1 and x0+128..x0+131) are a short extra pass.  All trip counts are compile-time.
    static_assert(RGROUPS == 34 && TW == 128, "stage 1 mapping");
    auto convert_group = [&](int ry, int gx, bool store_y) {
        const uint32_t* rw = s.rgb + ry * RWORDS + 3 * (gx + SKIP / 4);
        const uint32_t w0 = rw[0], w1 = rw[1], w2 = rw[2];
        const uint32_t px[4] = {w0, __funnelshift_r(w0, w1, 24), __funnelshift_r(w1, w2, 16), w2 >> 8};
        uint32_t yv[4], crv[4], cbv[4];          // results in byte 2
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t acc = __dp2a_hi(W_B, px[k], __dp2a_lo(W_RG, px[k], 4u * 8192u));
            const uint32_t yy = acc >> 16;
            yv[k] = acc;
            crv[k] = min(__dp2a_lo(K_CR, px[k], C4 - K_CR * yy), 0x00FFFFFFu);
            cbv[k] = __dp2a_hi(K_CB, px[k], C4 - K_CB * yy);
        }
        *reinterpret_cast<uint32_t*>(&s.cr[ry][4 * gx]) =
            __byte_perm(__byte_perm(crv[0], crv[1], 0x0062), __byte_perm(crv[2], crv[3], 0x0062), 0x5410);
        *reinterpret_cast<uint32_t*>(&s.cb[ry][4 * gx]) =
            __byte_perm(__byte_perm(cbv[0], cbv[1], 0x0062), __byte_perm(cbv[2], cbv[3], 0x0062), 0x5410);
        if (store_y)
            *reinterpret_cast<uint32_t*>(&s.y[ry - 2][4 * (gx - 1)]) =
                __byte_perm(__byte_perm(yv[0], yv[1], 0x0062), __byte_perm(yv[2], yv[3], 0x0062), 0x5410);
    };
    {
        const int warp = tid >> 5, lane = tid & 31;
#pragma unroll
        for (int k = 0; k < (RH + WARPS - 1) / WARPS; ++k) {
            const int ry = warp + WARPS * k;
            if (ry < RH) {
                wait_chunk(ry / CHUNK_ROWS);
                convert_group(ry, lane + 1, ry >= 2 && ry < 2 + TH);
            }
        }
#pragma unroll
        for (int c = 0; c < LOAD_CHUNKS; ++c) wait_chunk(c);
#pragma unroll
        for (int k = 0; k < (2 * RH + THREADS - 1) / THREADS; ++k) {
            const int i = tid + THREADS * k;
            if (i < 2 * RH) convert_group(i >> 1, (i & 1) ? RGROUPS - 1 : 0, false);
        }
    }
    __syncthreads();

    // ---- stage 2a: horizontal [1 4 6 4 1] at stride 2; chroma column cx reads region pixels 2 cx + 2 .. 2 cx + 6 ----
    // 16 four-output groups per row: R16 rows per step, one channel after the other
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
        for (int k = 0; k < (RH + R16 - 1) / R16; ++k) {
            const int ry = (tid >> 4) + R16 * k, j = tid & 15;
            if (ry < RH) {
                // (two 8-byte loads: a half-warp's 16 lanes cover one row's 128 bytes without a bank conflict; four
                // 4-byte loads of the two rows a warp works on collide pairwise)
                const uint2* row = reinterpret_cast<const uint2*>(ch == 0 ? s.cr[ry] : s.cb[ry]) + j;
                const uint2 lo = row[0], hi = row[1];
                const uint32_t wa = lo.x, wb = lo.y, wc = hi.x, wd = hi.y;
                const uint32_t o0 = __dp4a(wb, 0x00010406u, __dp4a(wa, 0x04010000u, 0u));
                const uint32_t o1 = __dp4a(wc, 0x00000001u, __dp4a(wb, 0x04060401u, 0u));
                const uint32_t o2 = __dp4a(wc, 0x00010406u, __dp4a(wb, 0x04010000u, 0u));
                const uint32_t o3 = __dp4a(wd, 0x00000001u, __dp4a(wc, 0x04060401u, 0u));
                *reinterpret_cast<uint2*>(&s.hpass[ch][ry][4 * j]) =
                    make_uint2(__byte_perm(o0, o1, 0x5410), __byte_perm(o2, o3, 0x5410));
            }
        }
    }
    __syncthreads();
    // ---- stage 2b: vertical on two 16-bit lanes per word (sums stay below 2^16), (sum + 128) >> 8.  A thread
    // makes two consecutive output rows from seven loads (the rows they share are loaded once) ----
    static_assert(CH % 2 == 0 && 2 * CH + 2 < RH + 1, "row pairs of stage 2b");
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
#pragma unroll
        for (int k = 0; k < (CH / 2 + R16 - 1) / R16; ++k) {
            const int cp = (tid >> 4) + R16 * k, j = tid & 15;
            if (cp < CH / 2) {
                uint2 t[7];
#pragma unroll
                for (int q = 0; q < 7; ++q) t[q] = *reinterpret_cast<const uint2*>(&s.hpass[ch][4 * cp + q][4 * j]);
                const uint32_t a0 = 0x00800080u + t[0].x + 4u * t[1].x + 6u * t[2].x + 4u * t[3].x + t[4].x;
                const uint32_t a1 = 0x00800080u + t[0].y + 4u * t[1].y + 6u * t[2].y + 4u * t[3].y + t[4].y;
                const uint32_t b0 = 0x00800080u + t[2].x + 4u * t[3].x + 6u * t[4].x + 4u * t[5].x + t[6].x;
                const uint32_t b1 = 0x00800080u + t[2].y + 4u * t[3].y + 6u * t[4].y + 4u * t[5].y + t[6].y;
                uint8_t (*dstp)[CD_PITCH] = ch == 0 ? s.crd : s.cbd;
                *reinterpret_cast<uint32_t*>(&dstp[2 * cp][4 * j]) = __byte_perm(a0, a1, 0x7531);       // the high byte of each 16-bit lane
                *reinterpret_cast<uint32_t*>(&dstp[2 * cp + 1][4 * j]) = __byte_perm(b0, b1, 0x7531);
            }
        }
    }
    __syncthreads();
    // ---- stage 2c (edge tiles only): samples outside the planes become 128, i.e. zero after the level
    // shift -- the reference zero-pads after x - 128 (transform.py:186-188).  Only the part of the tile past
    // the plane is visited. ----
    {
        const int vy = min(TH, h - y0), vx = min(TW, w - x0);                          // valid rows / columns of the tiles
        const int vcy = min(CH, g.hc - y0 / 2), vcx = min(CW, g.wc - x0 / 2);
        if (vy < TH || vx < TW || vcy < CH || vcx < CW) {
            const int ry0 = max(vy, 0), rc0 = max(vcy, 0);
            for (int i = tid; i < (TH - ry0) * (TW / 4); i += THREADS)                 // whole rows below the plane
                *reinterpret_cast<uint32_t*>(&s.y[ry0 + i / (TW / 4)][4 * (i % (TW / 4))]) = 0x80808080u;
            for (int i = tid; i < (CH - rc0) * (CW / 4); i += THREADS) {
                *reinterpret_cast<uint32_t*>(&s.crd[rc0 + i / (CW / 4)][4 * (i % (CW / 4))]) = 0x80808080u;
                *reinterpret_cast<uint32_t*>(&s.cbd[rc0 + i / (CW / 4)][4 * (i % (CW / 4))]) = 0x80808080u;
            }
            if (vx < TW) {                                                              // columns right of the plane
                const int c0 = max(vx, 0), nc = TW - c0;
                for (int i = tid; i < ry0 * nc; i += THREADS) s.y[i / nc][c0 + i % nc] = 128;
            }
            if (vcx < CW) {
                const int c0 = max(vcx, 0), nc = CW - c0;
                for (int i = tid; i < rc0 * nc; i += THREADS) {
                    s.crd[i / nc][c0 + i % nc] = 128;
                    s.cbd[i / nc][c0 + i % nc] = 128;
                }
            }
            __syncthreads();
        }
    }

    // ---- stage 3: the 8x8 blocks ----
    unsigned fl = 0;
    {
        TileBlock t;
        if (tile_block(tid, blockIdx.x, blockIdx.y, img, g, h, w, t)) {   // (false only for blocks past the plane, at the bottom / right edge)
            const uint8_t* pa = t.kind == 0 ? &s.y[8 * t.by][8 * t.bx] : (t.plane == 0 ? &s.crd[8 * t.by][8 * t.bx] : &s.cbd[8 * t.by][8 * t.bx]);
            const int pitch = t.kind == 0 ? TW : CD_PITCH;
            uint32_t wv[16];
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const uint2 v = *reinterpret_cast<const uint2*>(pa + r * pitch);
                wv[2 * r] = v.x;
                wv[2 * r + 1] = v.y;
            }
            fl = transform_single(t.kind, wv, &s.stage[tid * 8], tid & 7, t.rows, t.cols);
        }
    }
    // the warps are whole (luminance and chroma threads never share one) and converged again here
    const unsigned m = __ballot_sync(0xffffffffu, fl != 0);
    if ((tid & 31) == 0)
        flagmap[(((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x) * WARPS + (tid >> 5)] = m;
    // ---- stage 4: the staged blocks leave through TMA: the tile's luminance blocks as one box, its Cr and
    // Cb blocks as another; blocks past the planes are clipped by the tensor bounds ----
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
        const int lx = blockIdx.x * (TW / 8), ly = blockIdx.y * (TH / 8);
        const int cx = blockIdx.x * (CW / 8), cy = blockIdx.y * (CH / 8);
        if (lx < g.nbx_l && ly < g.nby_l)
            asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4}], [%5];"
                         ::"l"(reinterpret_cast<uint64_t>(&tmap_l)), "r"(0), "r"(lx), "r"(ly), "r"(img), "r"(smem_u32(s.stage))
                         : "memory");
        if (cx < g.nbx_c && cy < g.nby_c)
            asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%1, %2, %3, %4, %5}], [%6];"
                         ::"l"(reinterpret_cast<uint64_t>(&tmap_c)), "r"(0), "r"(cx), "r"(cy), "r"(0), "r"(img),
                         "r"(smem_u32(&s.stage[NY_BLOCKS * 8]))
                         : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");       // the staging area must outlive the reads
    }
}

// Float64 re-evaluation of every flagged block with scipy's exact operation order.  A warp takes FOUR
// flagged blocks at a time: all 32 lanes rebuild each block's samples from the RGB source in turn (for a
// chroma block the 19x19 window of Cr or Cb values, then the separable [1 4 6 4 1] pyramid); then every
// group of eight lanes runs its own block's eight row transforms, then its eight column transforms +
// quantisation, and corrects the float32 result in place -- the float64 passes are the long part, and
// with one block per warp 24 of the 32 lanes sat idle in them.
constexpr int FIX_WARPS = 8;
constexpr int FIX_GROUP = 4;      // blocks per warp
struct FixSmem {
    double a[64];                 // row-transformed block
    int16_t px[64];               // x - 128, zero padded
    uint16_t hp[19][8];           // horizontal pass of the chroma window
    uint8_t win[19][20];          // Cr or Cb of the 19x19 source window
};
struct FixBlock {                 // where a flagged block sits
    int kind, ph, pw, BY, BX, plane;
    int64_t img;
};
__device__ __forceinline__ FixBlock fix_locate(uint32_t block, const hic_dct_geometry& g, int h, int w) {
    FixBlock f;
    f.img = block / g.blocks_per_image;
    int64_t local = block - f.img * g.blocks_per_image;
    if (local < g.nb_l) {
        f.kind = 0; f.ph = h; f.pw = w; f.plane = 0;
        f.BY = (int)(local / g.nbx_l); f.BX = (int)(local % g.nbx_l);
    } else {
        f.kind = 1; f.ph = g.hc; f.pw = g.wc;
        local -= g.nb_l;
        f.plane = (int)(local / g.nb_c);
        local -= (int64_t)f.plane * g.nb_c;
        f.BY = (int)(local / g.nbx_c); f.BX = (int)(local % g.nbx_c);
    }
    return f;
}

__global__ void __launch_bounds__(32 * FIX_WARPS)
fixup_kernel(const uint8_t* __restrict__ rgb, int h, int w, hic_dct_geometry g, int16_t* __restrict__ coef,
             const hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    __shared__ FixSmem sm_all[FIX_WARPS][FIX_GROUP];
    const int lane = threadIdx.x & 31;
    const int grp = lane >> 3, l8 = lane & 7;
    const uint32_t n_rec = min(stats[0], tie_capacity);
    const uint32_t warps = gridDim.x * FIX_WARPS;
    uint32_t changed_total = 0, done = 0;
    for (uint32_t base = (blockIdx.x * FIX_WARPS + (threadIdx.x >> 5)) * FIX_GROUP; base < n_rec; base += warps * FIX_GROUP) {
        // ---- all lanes: the samples of each of the (up to) four blocks ----
        for (int k = 0; k < FIX_GROUP && base + k < n_rec; ++k) {
            FixSmem& sm = sm_all[threadIdx.x >> 5][k];
            const FixBlock f = fix_locate(ties[base + k].block, g, h, w);
            const uint8_t* src = rgb + (size_t)f.img * h * w * 3;
            if (f.kind == 0) {
                for (int e = lane; e < 64; e += 32) {
                    const int y = 8 * f.BY + (e >> 3), x = 8 * f.BX + (e & 7);
                    int val = 0;
                    if (y < h && x < w) {
                        const uint8_t* p = src + ((size_t)y * w + x) * 3;
                        int yy, cr, cb;
                        rgb_to_ycrcb(p[0], p[1], p[2], yy, cr, cb);
                        val = yy - 128;
                    }
                    sm.px[e] = (int16_t)val;
                }
            } else {
                const int y0 = 16 * f.BY - 2, x0 = 16 * f.BX - 2;        // window origin in the source image
                for (int e = lane; e < 19 * 19; e += 32) {
                    const int r = e / 19, c = e - r * 19;
                    const int y = reflect101(y0 + r, h), x = reflect101(x0 + c, w);
                    const uint8_t* p = src + ((size_t)y * w + x) * 3;
                    int yy, cr, cb;
                    rgb_to_ycrcb(p[0], p[1], p[2], yy, cr, cb);
                    sm.win[r][c] = (uint8_t)(f.plane == 0 ? cr : cb);
                }
                __syncwarp();
                for (int e = lane; e < 19 * 8; e += 32) {            // horizontal [1 4 6 4 1] at stride 2
                    const int r = e >> 3, c = e & 7;
                    const uint8_t* q = &sm.win[r][2 * c];
                    sm.hp[r][c] = (uint16_t)(q[0] + 4 * q[1] + 6 * q[2] + 4 * q[3] + q[4]);
                }
                __syncwarp();
                for (int e = lane; e < 64; e += 32) {                // vertical, (sum + 128) >> 8
                    const int r = e >> 3, c = e & 7;
                    int val = 0;
                    if (8 * f.BY + r < g.hc && 8 * f.BX + c < g.wc) {
                        const int sum = sm.hp[2 * r][c] + 4 * sm.hp[2 * r + 1][c] + 6 * sm.hp[2 * r + 2][c] +
                                        4 * sm.hp[2 * r + 3][c] + sm.hp[2 * r + 4][c];
                        val = ((sum + 128) >> 8) - 128;
                    }
                    sm.px[e] = (int16_t)val;
                }
            }
        }
        __syncwarp();
        // ---- eight lanes per block: rows, then columns ----
        const bool mine = base + grp < n_rec;
        FixSmem& sm = sm_all[threadIdx.x >> 5][grp];
        if (mine) {                                              // rows (transform.py:78-80)
            double row[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) row[j] = (double)sm.px[8 * l8 + j];
            ducc_dct2_8(row);
#pragma unroll
            for (int j = 0; j < 8; ++j) sm.a[8 * l8 + j] = row[j];
        }
        __syncwarp();
        uint32_t changed = 0;
        if (mine) {                                              // columns, division by the table, np.round
            const uint32_t block = ties[base + grp].block;
            const FixBlock f = fix_locate(block, g, h, w);
            double col[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) col[r] = sm.a[8 * r + l8];
            ducc_dct2_8(col);
            int16_t* blk = coef + (size_t)block * 64;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int nat = 8 * r + l8;
                if (nat == 0) continue;                          // DC is an exact integer in float32 too
                int32_t v = round_half_even(ddiv(col[r], (double)c_tab.qi[f.kind][nat]));
                // coefficients outside the unpadded plane stay zero (transform.py:63, codec.py:288)
                if (8 * f.BY + r >= f.ph || 8 * f.BX + l8 >= f.pw) v = 0;
                const int k = c_tab.izz[nat];
                if ((int32_t)blk[k] != v) {
                    blk[k] = (int16_t)v;
                    ++changed;
                }
            }
            if (l8 == 0) ++done;
        }
        changed_total += changed;
        __syncwarp();
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        changed_total += __shfl_down_sync(0xffffffffu, changed_total, off);
        done += __shfl_down_sync(0xffffffffu, done, off);
    }
    if (lane == 0) {
        if (done) atomicAdd(&stats[1], 63u * done);
        if (changed_total) atomicAdd(&stats[2], changed_total);
    }
}

}  // namespace k1

// ------------------------------------------------------------------------------------------------
// K7: dequantise + IDCT + 128 + uint8 cast, one 8x8 block per thread
// ------------------------------------------------------------------------------------------------
namespace k7 {
constexpr float MAGIC = 12582912.0f;

__device__ __forceinline__ void record_tie(uint32_t block, hic_tie_record* __restrict__ ties, uint32_t tie_capacity,
                                           uint32_t* __restrict__ stats) {
    const uint32_t slot = atomicAdd(&stats[0], 1u);
    if (slot < tie_capacity) {
        hic_tie_record rec;
        rec.block = block;
        rec.reserved = 0;
        rec.mask = ~0ull;
        ties[slot] = rec;
    } else {
        atomicAdd(&stats[3], 1u);
    }
}

// in: the block's 128-byte row of the staging area (TMA 128-byte swizzle: piece j sits at position j ^ sw)
template <int KIND>
__device__ __forceinline__ void inverse_block(const int4* __restrict__ in, int sw, uint8_t* __restrict__ plane, int ph,
                                              int pw, int BY, int BX, uint32_t block_index,
                                              hic_tie_record* __restrict__ ties, uint32_t tie_capacity,
                                              uint32_t* __restrict__ stats) {
    constexpr uint8_t zz[64] = HIC_ZIGZAG8;
    float v[64];
    float energy = 0.f;          // sum |coef * q| * w: the error band of the samples
    int ac_bits = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int4 wv = in[j ^ sw];
        const int words[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int k0 = 8 * j + 2 * e;
            const int lo = (int)(short)(words[e] & 0xFFFF), hi = words[e] >> 16;
            const float flo = (float)lo, fhi = (float)hi;
            v[zz[k0]] = flo * c_tab.dq[KIND][zz[k0]];
            v[zz[k0 + 1]] = fhi * c_tab.dq[KIND][zz[k0 + 1]];
            energy = fmaf(fabsf(flo), c_tab.qw[KIND][zz[k0]], energy);
            energy = fmaf(fabsf(fhi), c_tab.qw[KIND][zz[k0 + 1]], energy);
            ac_bits |= k0 == 0 ? (words[e] & 0xFFFF0000) : words[e];
        }
    }
#pragma unroll
    for (int r = 0; r < 8; ++r)
        eo_inverse8(v[8 * r + 0], v[8 * r + 1], v[8 * r + 2], v[8 * r + 3], v[8 * r + 4], v[8 * r + 5],
                    v[8 * r + 6], v[8 * r + 7]);
#pragma unroll
    for (int c = 0; c < 8; ++c)
        eo_inverse8(v[c], v[8 + c], v[16 + c], v[24 + c], v[32 + c], v[40 + c], v[48 + c], v[56 + c]);
    const int rows = min(8, ph - 8 * BY), cols = min(8, pw - 8 * BX);
    // distance of every sample to the nearest integer, where the reference's uint8 truncation steps
    float margin = 1e30f;
#pragma unroll
    for (int i = 0; i < 64; ++i) {
        v[i] += 128.f;
        const float r = (v[i] + MAGIC) - MAGIC;
        margin = fminf(margin, fabsf(v[i] - r));
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        if (r >= rows) break;
        uint32_t w0 = 0, w1 = 0;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const uint32_t b = (uint32_t)(__float2int_rz(v[8 * r + c])) & 0xFFu;   // truncate, wrap
            if (c < 4) w0 |= b << (8 * c); else w1 |= b << (8 * (c - 4));
        }
        uint8_t* dst = plane + (size_t)(8 * BY + r) * pw + 8 * BX;
        if (cols == 8 && ((reinterpret_cast<uintptr_t>(dst) & 7) == 0)) {
            *reinterpret_cast<uint2*>(dst) = make_uint2(w0, w1);
        } else {
            for (int c = 0; c < cols; ++c) dst[c] = (uint8_t)((c < 4 ? w0 >> (8 * c) : w1 >> (8 * (c - 4))) & 0xFF);
        }
    }
    // a DC-only block is exact in both float32 and float64 (no rounding happens at all)
    // energy = sum |coef| q w(u, v) margin: the rigorous per-input error weights of hic_dct_bound.h; 2^-15 covers the
    // rounding of the final + 128 (half an ulp of a value below 512) and of this comparison
    const float band = (float)(4.0 / 16777216.0 / 256.0) * energy + 3.0517578125e-5f;
    if (ac_bits != 0 && margin <= band) record_tie(block_index, ties, tie_capacity, stats);
}

// One TMA tensor load of the CTA's box of K7's [block][64 int16] map (box_rows blocks from block blockIdx.x * box_rows)
// into dst (bytes long): thread 0 issues it on the mbarrier bar, and every thread returns once it has landed.
__device__ __forceinline__ void load_block_box(const CUtensorMap& tmap, int box_rows, void* dst, uint32_t bytes,
                                               unsigned long long* bar_p) {
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(bar_p);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
            ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(0),
            "r"((int)(blockIdx.x * box_rows)), "r"(bar)
            : "memory");
    }
    __syncthreads();
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}\n" ::"r"(bar)
        : "memory");
}

// Global block index b of the batch (per image its Y blocks, then Cr, then Cb, each row by row): its image, plane p
// (0 = Y, 1 = Cr, 2 = Cb) and block row and column in that plane.
struct BlockPos {
    int64_t img;
    int p, by, bx;
};
__device__ __forceinline__ BlockPos block_pos(const hic_dct_geometry& g, int64_t b) {
    BlockPos q;
    q.img = b / g.blocks_per_image;
    int64_t local = b - q.img * g.blocks_per_image;
    int nbx = g.nbx_l;
    q.p = 0;
    if (local >= g.nb_l) {
        local -= g.nb_l;
        q.p = 1;
        if (local >= g.nb_c) {
            local -= g.nb_c;
            q.p = 2;
        }
        nbx = g.nbx_c;
    }
    q.by = (int)(local / nbx);
    q.bx = (int)(local % nbx);
    return q;
}

// A CTA takes K7_THREADS consecutive blocks of the coefficient buffer: ONE TMA tensor load (the buffer as
// [block][64 int16], box {64, K7_THREADS}, 128-byte swizzle) brings their 16 KB into shared memory, and a
// thread reads its own block from there with conflict-free 16-byte loads.  (A thread loading its 128-byte
// line straight from global memory is a load of 32 different lines per warp instruction -- the same LSU
// wavefront bill K1's stores used to pay.)
constexpr int K7_THREADS = 128;
struct K7Smem {
    alignas(1024) int4 blk[K7_THREADS * 8];
    alignas(8) unsigned long long bar;
};

__global__ void __launch_bounds__(K7_THREADS)
inverse_kernel(const __grid_constant__ CUtensorMap tmap_blocks, hic_dct_geometry g, int n, uint8_t* __restrict__ yp,
               uint8_t* __restrict__ crp, uint8_t* __restrict__ cbp, hic_tie_record* __restrict__ ties,
               uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    __shared__ K7Smem s;
    load_block_box(tmap_blocks, K7_THREADS, s.blk, sizeof(s.blk), &s.bar);
    const int64_t total = (int64_t)n * g.blocks_per_image;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= total) return;
    const int64_t img = gid / g.blocks_per_image;
    int64_t local = gid - img * g.blocks_per_image;
    const int4* src = &s.blk[threadIdx.x * 8];
    const int sw = threadIdx.x & 7;
    if (local < g.nb_l) {
        inverse_block<0>(src, sw, yp + (size_t)img * g.h * g.w, g.h, g.w, (int)(local / g.nbx_l), (int)(local % g.nbx_l),
                         (uint32_t)gid, ties, tie_capacity, stats);
    } else {
        local -= g.nb_l;
        const int plane = (int)(local / g.nb_c);
        local -= (int64_t)plane * g.nb_c;
        uint8_t* base = (plane == 0 ? crp : cbp) + (size_t)img * g.hc * g.wc;
        inverse_block<1>(src, sw, base, g.hc, g.wc, (int)(local / g.nbx_c), (int)(local % g.nbx_c), (uint32_t)gid, ties,
                         tie_capacity, stats);
    }
}

// Where a flagged block's samples go: the plane (row stride pw, ph rows) and the block's position in it.
struct BlockDst {
    uint8_t* plane;
    int ph, pw, BY, BX;
};

// Float64 re-evaluation of every flagged sample with scipy's exact operation order.  locate(img, p, BY, BX) maps
// block (BY, BX) of plane p (0 = Y, 1 = Cr, 2 = Cb) of image img to its BlockDst.
template <class Locate>
__device__ __forceinline__ void inverse_fixup_body(const int16_t* __restrict__ coef, const hic_dct_geometry& g,
                                                   const hic_tie_record* __restrict__ ties, uint32_t tie_capacity,
                                                   uint32_t* __restrict__ stats, Locate locate) {
    // eight lanes per flagged block (four blocks per warp): lane r runs the block's row r, then its column
    // r, in exact_decoded_block's order (rows first, then columns, /256, +128); the row results cross the
    // lanes through shared memory
    __shared__ double s_a[4][4][64];                 // [warp][block of the warp][row-transformed block]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, l8 = lane & 7;
    const uint32_t n_rec = min(stats[0], tie_capacity);
    const uint32_t groups = gridDim.x * (blockDim.x / 8);
    uint32_t changed_total = 0, done = 0;
    for (uint32_t base = (blockIdx.x * (blockDim.x / 32) + warp) * 4; base < n_rec; base += groups) {
        const uint32_t i = base + grp;
        const bool mine = i < n_rec;
        double* a = s_a[warp][grp];
        int kind = 0, nbx = g.nbx_l;
        BlockDst d = {nullptr, 0, 0, 0, 0};
        if (mine) {
            const hic_tie_record rec = ties[i];
            const int64_t img = rec.block / g.blocks_per_image;
            int64_t local = rec.block - img * g.blocks_per_image;
            int p = 0;
            if (local >= g.nb_l) {
                kind = 1;
                local -= g.nb_l;
                p = (int)(local / g.nb_c);
                local -= (int64_t)p * g.nb_c;
                nbx = g.nbx_c;
                ++p;
            }
            d = locate(img, p, (int)(local / nbx), (int)(local % nbx));
            const int16_t* blk = coef + (size_t)rec.block * 64;
            double row[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int nat = 8 * l8 + j;
                row[j] = (double)((int32_t)blk[c_tab.izz[nat]] * c_tab.qi[kind][nat]);
            }
            ducc_dct3_8(row);
#pragma unroll
            for (int j = 0; j < 8; ++j) a[8 * l8 + j] = row[j];
        }
        __syncwarp();
        if (mine) {
            double col[8];
#pragma unroll
            for (int r = 0; r < 8; ++r) col[r] = a[8 * r + l8];
            ducc_dct3_8(col);
            uint32_t changed = 0;
#pragma unroll
            for (int y = 0; y < 8; ++y) {
                if (8 * d.BY + y >= d.ph || 8 * d.BX + l8 >= d.pw) continue;
                const uint8_t v = wrap_u8(dadd(ddiv(col[y], 256.0), 128.0));
                uint8_t* dst = d.plane + (size_t)(8 * d.BY + y) * d.pw + 8 * d.BX + l8;
                if (*dst != v) {
                    *dst = v;
                    ++changed;
                }
            }
            changed_total += changed;
            if (l8 == 0) ++done;
        }
        __syncwarp();
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        changed_total += __shfl_down_sync(0xffffffffu, changed_total, off);
        done += __shfl_down_sync(0xffffffffu, done, off);
    }
    if (lane == 0) {
        if (done) atomicAdd(&stats[1], 64u * done);
        if (changed_total) atomicAdd(&stats[2], changed_total);
    }
}

__global__ void __launch_bounds__(128)
inverse_fixup_kernel(const int16_t* __restrict__ coef, hic_dct_geometry g, uint8_t* __restrict__ yp,
                     uint8_t* __restrict__ crp, uint8_t* __restrict__ cbp, const hic_tie_record* __restrict__ ties,
                     uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    inverse_fixup_body(coef, g, ties, tie_capacity, stats, [&](int64_t img, int p, int BY, int BX) {
        if (p == 0) return BlockDst{yp + (size_t)img * g.h * g.w, g.h, g.w, BY, BX};
        return BlockDst{(p == 1 ? crp : cbp) + (size_t)img * g.hc * g.wc, g.hc, g.wc, BY, BX};
    });
}

// K8's pyrUp neighbours of sample i on an axis of n samples: i - 1 and i + 1, with s[-1] = s[1] and s[n] = s[n-1]
__device__ __forceinline__ void pyr_neighbours(int i, int n, int& prev, int& next) {
    prev = i > 0 ? i - 1 : (n > 1 ? 1 : 0);
    next = i + 1 < n ? i + 1 : n - 1;
}

// K8's pyrUp of one chroma sample's 2x2 output quad [2 dy + dx] from its 3x3 neighbourhood: r0, r1, r2 the rows
// ym, cy, yn, each at columns xm, cx, xn (pyr_neighbours).  Per axis even = s[i-1] + 6 s[i] + s[i+1], odd =
// 4 (s[i] + s[i+1]); (v + 32) >> 6 after both axes.
__device__ __forceinline__ void pyr_up_quad(const int* r0, const int* r1, const int* r2, int* up) {
    const int e0 = r0[0] + 6 * r0[1] + r0[2], o0 = 4 * (r0[1] + r0[2]);
    const int e1 = r1[0] + 6 * r1[1] + r1[2], o1 = 4 * (r1[1] + r1[2]);
    const int e2 = r2[0] + 6 * r2[1] + r2[2], o2 = 4 * (r2[1] + r2[2]);
    up[0] = (e0 + 6 * e1 + e2 + 32) >> 6;
    up[1] = (o0 + 6 * o1 + o2 + 32) >> 6;
    up[2] = (4 * (e1 + e2) + 32) >> 6;
    up[3] = (4 * (o1 + o2) + 32) >> 6;
}

// K8's ycrcb_to_rgb of one pixel, written to o[0..2]
__device__ __forceinline__ void store_rgb(uint8_t* o, int y, int cr, int cb) {
    int r, gg, b;
    ycrcb_to_rgb(y, cr, cb, r, gg, b);
    o[0] = (uint8_t)r;
    o[1] = (uint8_t)gg;
    o[2] = (uint8_t)b;
}

// K8: cv2.pyrUp of both chroma planes + crop + YCrCb -> RGB.  One thread per chroma sample, producing the 2x2 output
// quad through pyr_up_quad.
__global__ void __launch_bounds__(256)
upsample_colour_kernel(const uint8_t* __restrict__ yp, const uint8_t* __restrict__ crp,
                       const uint8_t* __restrict__ cbp, hic_dct_geometry g, int n, uint8_t* __restrict__ rgb) {
    const int64_t per = (int64_t)g.hc * g.wc;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    const int cy = (int)(rem / g.wc), cx = (int)(rem % g.wc);
    int ym, yn, xm, xn;
    pyr_neighbours(cy, g.hc, ym, yn);
    pyr_neighbours(cx, g.wc, xm, xn);
    int up[2][4];      // [channel][2*dy + dx]
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
        const uint8_t* p = (ch == 0 ? crp : cbp) + (size_t)img * per;
        const int r0[3] = {p[(size_t)ym * g.wc + xm], p[(size_t)ym * g.wc + cx], p[(size_t)ym * g.wc + xn]};
        const int r1[3] = {p[(size_t)cy * g.wc + xm], p[(size_t)cy * g.wc + cx], p[(size_t)cy * g.wc + xn]};
        const int r2[3] = {p[(size_t)yn * g.wc + xm], p[(size_t)yn * g.wc + cx], p[(size_t)yn * g.wc + xn]};
        pyr_up_quad(r0, r1, r2, up[ch]);
    }
    const uint8_t* ysrc = yp + (size_t)img * g.h * g.w;
    uint8_t* dst = rgb + (size_t)img * g.out_h * g.out_w * 3;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int oy = 2 * cy + dy, ox = 2 * cx + dx;
            int r, gg, b;
            ycrcb_to_rgb(ysrc[(size_t)oy * g.w + ox], up[0][2 * dy + dx], up[1][2 * dy + dx], r, gg, b);
            uint8_t* o = dst + ((size_t)oy * g.out_w + ox) * 3;
            o[0] = (uint8_t)r;
            o[1] = (uint8_t)gg;
            o[2] = (uint8_t)b;
        }
}

// The same, four chroma samples (8 x 2 output pixels) per thread with word loads and stores: used when
// the rows are word aligned (wc % 4 == 0, which makes w % 8 == 0 and out_w * 3 % 4 == 0).
__global__ void __launch_bounds__(256)
upsample_colour_vec_kernel(const uint8_t* __restrict__ yp, const uint8_t* __restrict__ crp,
                           const uint8_t* __restrict__ cbp, hic_dct_geometry g, int n, uint8_t* __restrict__ rgb) {
    const int groups = g.wc / 4;
    const int64_t per = (int64_t)g.hc * groups;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    const int cy = (int)(rem / groups), cx = 4 * (int)(rem % groups);
    int ym, yn;
    pyr_neighbours(cy, g.hc, ym, yn);
    int up[2][2][8];          // [channel][output row parity][output column]
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
        const uint8_t* p = (ch == 0 ? crp : cbp) + (size_t)img * g.hc * g.wc;
        int hrow[3][8];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const uint8_t* q = p + (size_t)(r == 0 ? ym : (r == 1 ? cy : yn)) * g.wc;
            const uint32_t mid = __ldg(reinterpret_cast<const uint32_t*>(q + cx));
            int sv[6];
            sv[1] = mid & 0xFF; sv[2] = (mid >> 8) & 0xFF; sv[3] = (mid >> 16) & 0xFF; sv[4] = mid >> 24;
            sv[0] = cx > 0 ? (int)__ldg(q + cx - 1) : (g.wc > 1 ? sv[2] : sv[1]);          // s[-1] = s[1]
            sv[5] = cx + 4 < g.wc ? (int)__ldg(q + cx + 4) : sv[4];                          // s[n] = s[n-1]
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                hrow[r][2 * i] = sv[i] + 6 * sv[i + 1] + sv[i + 2];
                hrow[r][2 * i + 1] = 4 * (sv[i + 1] + sv[i + 2]);
            }
        }
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            up[ch][0][x] = (hrow[0][x] + 6 * hrow[1][x] + hrow[2][x] + 32) >> 6;
            up[ch][1][x] = (4 * (hrow[1][x] + hrow[2][x]) + 32) >> 6;
        }
    }
    const uint8_t* ysrc = yp + (size_t)img * g.h * g.w;
    uint8_t* dst = rgb + (size_t)img * g.out_h * g.out_w * 3;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
        const int oy = 2 * cy + dy, ox = 2 * cx;
        const uint2 yw = __ldg(reinterpret_cast<const uint2*>(ysrc + (size_t)oy * g.w + ox));
        uint8_t px[24];
#pragma unroll
        for (int x = 0; x < 8; ++x) {
            const int yy = (int)(((x < 4 ? yw.x : yw.y) >> (8 * (x & 3))) & 0xFF);
            int r, gg, b;
            ycrcb_to_rgb(yy, up[0][dy][x], up[1][dy][x], r, gg, b);
            px[3 * x] = (uint8_t)r;
            px[3 * x + 1] = (uint8_t)gg;
            px[3 * x + 2] = (uint8_t)b;
        }
        uint32_t* o = reinterpret_cast<uint32_t*>(dst + ((size_t)oy * g.out_w + ox) * 3);
#pragma unroll
        for (int k = 0; k < 6; ++k)
            o[k] = (uint32_t)px[4 * k] | ((uint32_t)px[4 * k + 1] << 8) | ((uint32_t)px[4 * k + 2] << 16) | ((uint32_t)px[4 * k + 3] << 24);
    }
}

// A block whose AC terms are all zero decodes (K7: q T00 through the IDCT, /256, +128, astype(uint8)) to one
// constant sample: trunc(q T00 / 256 + 128) mod 256 = ((q T00 + 32768) / 256, truncated toward zero) & 255.
__device__ __forceinline__ int dc_block_sample(int q, int t00) { return ((q * t00 + 32768) / 256) & 255; }

// Thumbnail: one pixel per 8x8 tile of the full decode's output (th = ceil(out_h / 8), tw = ceil(out_w / 8)),
// from the DC values alone (one int16 per block, global block order).  The luminance block (ty, tx) gives Y; the
// chroma planes of block samples (nby_c x nbx_c) go through K8's pyrUp taps on the fly, s[-1] = s[1] and s[n] =
// s[n-1] per axis, and are cropped to th x tw with Y; then K8's ycrcb_to_rgb.  One thread per thumbnail pixel.
// thumbnail_pixel: pixel (ty, tx) of one image (blocks: its DC values) to o[0..2].
__device__ __forceinline__ void thumbnail_pixel(const int16_t* __restrict__ blocks, const hic_dct_geometry& g, int ty, int tx,
                                                uint8_t* __restrict__ o) {
    const int t_l = c_tab.qi[0][0], t_c = c_tab.qi[1][0];
    const int y = dc_block_sample(__ldg(blocks + (int64_t)ty * g.nbx_l + tx), t_l);
    const int cy = ty >> 1, cx = tx >> 1;
    const bool odd_y = ty & 1, odd_x = tx & 1;
    int ym, yn, xm, xn;
    pyr_neighbours(cy, g.nby_c, ym, yn);
    pyr_neighbours(cx, g.nbx_c, xm, xn);
    int up[2];
#pragma unroll
    for (int ch = 0; ch < 2; ++ch) {
        const int16_t* p = blocks + g.nb_l + ch * g.nb_c;
        auto s = [&](int r, int c) { return dc_block_sample(__ldg(p + (int64_t)r * g.nbx_c + c), t_c); };
        // horizontal pass on the rows the vertical tap needs, then the vertical tap
        auto hor = [&](int r) { return odd_x ? 4 * (s(r, cx) + s(r, xn)) : s(r, xm) + 6 * s(r, cx) + s(r, xn); };
        const int v = odd_y ? 4 * (hor(cy) + hor(yn)) : hor(ym) + 6 * hor(cy) + hor(yn);
        up[ch] = (v + 32) >> 6;
    }
    store_rgb(o, y, up[0], up[1]);
}

__global__ void __launch_bounds__(256)
thumbnail_kernel(const int16_t* __restrict__ dc, hic_dct_geometry g, int n, int th, int tw, uint8_t* __restrict__ rgb) {
    const int64_t per = (int64_t)th * tw;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    thumbnail_pixel(dc + img * g.blocks_per_image, g, (int)(rem / tw), (int)(rem % tw), rgb + gid * 3);
}

// The 1/8-scale window: one rh x rw window of the thumbnail per image, its origin (top, left) per image in thumbnail
// coordinates; one thread per window pixel, thumbnail_pixel straight from the DC values, n x rh x rw x 3 out.
__global__ void __launch_bounds__(256)
thumbnail_region_kernel(const int16_t* __restrict__ dc, hic_dct_geometry g, int n, const int32_t* __restrict__ origin, int rh,
                        int rw, uint8_t* __restrict__ rgb) {
    const int64_t per = (int64_t)rh * rw;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    const int top = __ldg(origin + 2 * img), left = __ldg(origin + 2 * img + 1);
    thumbnail_pixel(dc + img * g.blocks_per_image, g, top + (int)(rem / rw), left + (int)(rem % rw), rgb + gid * 3);
}

// ---- scaled decode: K7S, its fix-up, K8S (1/s scale, M = 8 / s samples per block side) ----------------------
// The work buffer holds one M x M tile of samples per block of the batch, in global block order: block b's samples
// at work + b M^2, row major.  K8S reads the reduced planes through that layout (r, c >= 0).
template <int M>
__device__ __forceinline__ int tile_sample(const uint8_t* plane, int nbx, unsigned r, unsigned c) {
    return plane[((r / M * nbx + c / M) * M + r % M) * M + c % M];
}

// The 16-byte pieces (8 scan entries each) of a block that the decode at M x M samples per block reads: all eight at
// M = 8; entries 0..31 at M = 4 (its 4 x 4 corner ends at entry 24); entries 0..7 at M = 2 (the 2 x 2 corner ends at 4).
template <int M>
constexpr int block_pieces() { return M == 8 ? 8 : (M == 4 ? 4 : 1); }

// Piece j of staged block t (16-byte units of a CTA's staging area): K7's 128-byte swizzle at M = 8 (j ^ (t & 7)),
// the 64-byte swizzle at M = 4 (j ^ ((t >> 1) & 3): the eight blocks of a quarter warp hit eight different 16-byte
// bank groups), none at M = 2.
template <int M>
__device__ __forceinline__ int staged_piece(int t, int j) {
    return block_pieces<M>() * t + (M == 8 ? j ^ (t & 7) : (M == 4 ? j ^ ((t >> 1) & 3) : j));
}

// K7S: one block per thread.  The CTA's 128 blocks arrive by one TMA tensor load over K7's [block][64 int16] map of
// the coefficient buffer, only the pieces the block needs (block_pieces): a box of {32, 128} in the 64-byte swizzle
// at M = 4, of {8, 128} at M = 2.  The float32 path is scaled_transform<M> on q T / 256 (exact); a block with AC
// terms and a sample within its band of an integer (where the uint8 truncation steps) is recorded for the float64
// fix-up.
constexpr int K7S_THREADS = 128;
template <int M>
struct K7SSmem {
    alignas(1024) int4 blk[K7S_THREADS * block_pieces<M>()];
    alignas(8) unsigned long long bar;
};

// K7S's arithmetic on staged block t of kind 0 (luminance) / 1 (chroma): its M x M tile, four samples per word, into
// packed; true when the block has AC terms and a sample within its error band of an integer.
template <int M>
__device__ __forceinline__ bool scaled_block(const int4* __restrict__ blk, int t, int kind, uint32_t (&packed)[M * M / 4]) {
    constexpr int PIECES = block_pieces<M>();
    constexpr uint8_t zz[64] = HIC_ZIGZAG8;
    int words[4 * PIECES];                              // the block's first 8 PIECES scan entries, two per word
#pragma unroll
    for (int j = 0; j < PIECES; ++j) {
        const int4 wv = blk[staged_piece<M>(t, j)];
        words[4 * j] = wv.x; words[4 * j + 1] = wv.y; words[4 * j + 2] = wv.z; words[4 * j + 3] = wv.w;
    }
    float v[M * M];
    float energy = 0.f;          // sum |q| T w_s margin: the error band of the samples
    int ac_bits = 0;
#pragma unroll
    for (int k = 0; k < 8 * PIECES; ++k) {
        const int nat = zz[k], u = nat >> 3, x = nat & 7;
        if (u >= M || x >= M) continue;
        const int q = (k & 1) ? words[k >> 1] >> 16 : (int)(short)(words[k >> 1] & 0xFFFF);
        v[M * u + x] = (float)(q * c_tab.qi[kind][nat]) * (1.f / 256.f);
        energy = fmaf(fabsf((float)q), c_tab.sqw[M == 4 ? 0 : 1][kind][M * u + x], energy);
        if (k) ac_bits |= q;
    }
    scaled_transform<M>(v);
    float margin = 1e30f;
#pragma unroll
    for (int i = 0; i < M * M; ++i) {
        const float p = v[i] + 128.f;
        const float r = (p + MAGIC) - MAGIC;
        margin = fminf(margin, fabsf(p - r));
        const uint32_t b = (uint32_t)__float2int_rz(p) & 0xFFu;               // truncate, wrap
        if (i % 4 == 0) packed[i / 4] = b; else packed[i / 4] |= b << (8 * (i % 4));
    }
    // as K7: 2^-15 covers the rounding of the final + 128 below 1024 and of this comparison
    const float band = (float)(4.0 / 16777216.0 / 256.0) * energy + 3.0517578125e-5f;
    return ac_bits != 0 && margin <= band;
}

template <int M>
__device__ __forceinline__ void store_tile(uint8_t* __restrict__ dst, const uint32_t (&packed)[M * M / 4]) {
    if constexpr (M == 4)
        *reinterpret_cast<uint4*>(dst) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
    else
        *reinterpret_cast<uint32_t*>(dst) = packed[0];
}

template <int M>
__global__ void __launch_bounds__(K7S_THREADS)
scaled_inverse_kernel(const __grid_constant__ CUtensorMap tmap_blocks, hic_dct_geometry g, int n, uint8_t* __restrict__ tiles,
                      hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    __shared__ K7SSmem<M> s;
    load_block_box(tmap_blocks, K7S_THREADS, s.blk, sizeof(s.blk), &s.bar);
    const int64_t total = (int64_t)n * g.blocks_per_image;
    const int64_t gid = (int64_t)blockIdx.x * K7S_THREADS + threadIdx.x;
    if (gid >= total) return;
    uint32_t packed[M * M / 4];
    const bool flagged = scaled_block<M>(s.blk, threadIdx.x, block_pos(g, gid).p == 0 ? 0 : 1, packed);
    store_tile<M>(tiles + gid * M * M, packed);
    if (flagged) record_tie((uint32_t)gid, ties, tie_capacity, stats);
}

// The fix-up of K7S's flagged blocks: one thread per record, scaled_decoded_block<M> (the float64 definition) into
// the block's tile, which locate(global block index) gives.  stats[1] counts the samples re-evaluated, stats[2] those
// that changed.
template <int M, class Locate>
__device__ __forceinline__ void scaled_fixup_body(const int16_t* __restrict__ coef, const hic_dct_geometry& g,
                                                  const hic_tie_record* __restrict__ ties, uint32_t tie_capacity,
                                                  uint32_t* __restrict__ stats, Locate locate) {
    const uint32_t n_rec = min(stats[0], tie_capacity);
    uint32_t changed = 0, done = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += gridDim.x * blockDim.x) {
        const uint32_t b = ties[i].block;
        const int kind = block_pos(g, b).p == 0 ? 0 : 1;
        const int16_t* blk = coef + (size_t)b * 64;
        int32_t cq[M * M];
#pragma unroll
        for (int u = 0; u < M; ++u)
#pragma unroll
            for (int x = 0; x < M; ++x) cq[M * u + x] = (int32_t)blk[c_tab.izz[8 * u + x]] * c_tab.qi[kind][8 * u + x];
        double y[M * M];
        scaled_decoded_block<M>(cq, y);
        uint8_t* dst = locate(b);
#pragma unroll
        for (int k = 0; k < M * M; ++k) {
            const uint8_t val = wrap_u8(y[k]);
            if (dst[k] != val) {
                dst[k] = val;
                ++changed;
            }
        }
        ++done;
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        changed += __shfl_down_sync(0xffffffffu, changed, off);
        done += __shfl_down_sync(0xffffffffu, done, off);
    }
    if ((threadIdx.x & 31) == 0) {
        if (done) atomicAdd(&stats[1], (uint32_t)(M * M) * done);
        if (changed) atomicAdd(&stats[2], changed);
    }
}

template <int M>
__global__ void __launch_bounds__(128)
scaled_fixup_kernel(const int16_t* __restrict__ coef, hic_dct_geometry g, uint8_t* __restrict__ tiles,
                    const hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    scaled_fixup_body<M>(coef, g, ties, tie_capacity, stats, [&](uint32_t b) { return tiles + (size_t)b * M * M; });
}

// The chroma planes (rows, columns) whose borders K8's taps reflect and replicate at, M samples per block side: the
// full decode's hc x wc at M = 8; the reduced planes' whole block grids, M nby_c x M nbx_c, below (the thumbnail's
// convention).  The two differ wherever hc or wc is not a multiple of 8.
template <int M>
__device__ __forceinline__ int2 chroma_extent(const hic_dct_geometry& g) {
    return M == 8 ? make_int2(g.hc, g.wc) : make_int2(M * g.nby_c, M * g.nbx_c);
}

// The pyrUp of chroma sample (cy, cx) of planes of ny x nx samples: the 2x2 quads up[c] of Cr (c = 0) and Cb (c = 1),
// from the 3x3 neighbourhood chosen with K8's borders in those planes and read through sample(c, row, col).
template <class Sample>
__device__ __forceinline__ void chroma_up_quads(int cy, int cx, int2 extent, Sample sample, int (&up)[2][4]) {
    int ym, yn, xm, xn;
    pyr_neighbours(cy, extent.x, ym, yn);
    pyr_neighbours(cx, extent.y, xm, xn);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        auto row = [&](int r, int* v) {
            v[0] = sample(c, r, xm); v[1] = sample(c, r, cx); v[2] = sample(c, r, xn);
        };
        int s0[3], s1[3], s2[3];
        row(ym, s0); row(cy, s1); row(yn, s2);
        pyr_up_quad(s0, s1, s2, up[c]);
    }
}

// K8S: one sample of the reduced chroma planes (chroma_extent) per thread, as K8: its 3x3 neighbourhood through
// pyr_up_quad, Y from the reduced luminance plane (M nby_l x M nbx_l), K8's ycrcb_to_rgb, and the pixels of its 2x2
// output quad inside sh x sw = ceil(out_h / s) x ceil(out_w / s) written to n x sh x sw x 3 directly.
template <int M>
__global__ void __launch_bounds__(256)
scaled_colour_kernel(const uint8_t* __restrict__ tiles, hic_dct_geometry g, int n, int sh, int sw, uint8_t* __restrict__ rgb) {
    const int qh = (sh + 1) / 2, qw = (sw + 1) / 2;
    const int64_t per = (int64_t)qh * qw;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    const int cy = (int)(rem / qw), cx = (int)(rem % qw);
    const uint8_t* base = tiles + (size_t)img * g.blocks_per_image * M * M;
    int up[2][4];
    chroma_up_quads(cy, cx, chroma_extent<M>(g), [&](int c, int r, int col) {
        return tile_sample<M>(base + (size_t)(g.nb_l + c * g.nb_c) * M * M, g.nbx_c, r, col);
    }, up);
    uint8_t* dst = rgb + (size_t)img * sh * sw * 3;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int oy = 2 * cy + dy, ox = 2 * cx + dx;
            if (oy >= sh || ox >= sw) continue;
            store_rgb(dst + ((size_t)oy * sw + ox) * 3, tile_sample<M>(base, g.nbx_l, oy, ox), up[0][2 * dy + dx],
                      up[1][2 * dy + dx]);
        }
}

// ---- region decode: K7R, its fix-up, K8R (one rh x rw window per image, its origin per image) ------------------
// One template per stage for M = 8 / s samples per block side: M = 8 is the window of the decoded image, M = 4 and 2
// the window of its 1/2- and 1/4-scale image.  The rectangles come from the region rules at M (region_first<M>,
// region_span<M>).  Image i's window-local tiles: Y at y + i * ly, the M x M tiles of the luminance rectangle's blocks,
// block row by block row (nx_l per row); Cr and Cb at cr / cb + i * lc likewise (nx_c per row).
struct RegionArgs {
    const int32_t* origin;      // n x (top, left), output coordinates (of the 1/scale image for the scaled decode)
    uint8_t *y, *cr, *cb;
    size_t ly, lc;
    RegionSpan s;
    int rh, rw;
};
struct RegionFirst {
    int by_l, bx_l, by_c, bx_c;
};
template <int M>
__device__ __forceinline__ RegionFirst region_first(const hic_dct_geometry& g, const RegionArgs& a, int64_t img) {
    const int top = __ldg(a.origin + 2 * img), left = __ldg(a.origin + 2 * img + 1);
    return {region_first_l<M>(top, a.s.ny_l, g.nby_l), region_first_l<M>(left, a.s.nx_l, g.nbx_l),
            region_first_c<M>(top, a.s.ny_c, g.nby_c), region_first_c<M>(left, a.s.nx_c, g.nbx_c)};
}

// Selected block `local` of image img (the nl luminance blocks of its rectangle row by row, then the nc of Cr, then
// Cb): its plane p (0 = Y, 1 = Cr, 2 = Cb), its place (ly, lx) in the rectangle, and its global block index.
template <int M>
__device__ __forceinline__ int64_t region_block(const hic_dct_geometry& g, const RegionArgs& a, int64_t img, int64_t local,
                                                int64_t nl, int64_t nc, int& p, int& ly, int& lx) {
    const RegionFirst f = region_first<M>(g, a, img);
    int64_t block = img * g.blocks_per_image;
    if (local < nl) {
        ly = (int)(local / a.s.nx_l);
        lx = (int)(local % a.s.nx_l);
        block += (int64_t)(f.by_l + ly) * g.nbx_l + f.bx_l + lx;
    } else {
        local -= nl;
        p = 1 + (int)(local / nc);
        local -= (int64_t)(p - 1) * nc;
        ly = (int)(local / a.s.nx_c);
        lx = (int)(local % a.s.nx_c);
        block += g.nb_l + (int64_t)(p - 1) * g.nb_c + (int64_t)(f.by_c + ly) * g.nbx_c + f.bx_c + lx;
    }
    return block;
}

template <int M>
__device__ __forceinline__ uint8_t* region_tile(const RegionArgs& a, int64_t img, int p, int ly, int lx) {
    if (p == 0) return a.y + img * a.ly + ((size_t)ly * a.s.nx_l + lx) * M * M;
    return (p == 1 ? a.cr : a.cb) + img * a.lc + ((size_t)ly * a.s.nx_c + lx) * M * M;
}

// Staged block t of plane p through K7's arithmetic (M = 8) or K7S's into its tile; a flagged block is recorded with
// its global block index `block`.
template <int M>
__device__ __forceinline__ void region_tile_block(const int4* __restrict__ blk, int t, int p, uint8_t* __restrict__ tile,
                                                  uint32_t block, hic_tie_record* __restrict__ ties, uint32_t tie_capacity,
                                                  uint32_t* __restrict__ stats) {
    if constexpr (M == 8) {
        if (p == 0)
            inverse_block<0>(blk + 8 * t, t & 7, tile, 8, 8, 0, 0, block, ties, tie_capacity, stats);
        else
            inverse_block<1>(blk + 8 * t, t & 7, tile, 8, 8, 0, 0, block, ties, tie_capacity, stats);
    } else {
        uint32_t packed[M * M / 4];
        const bool flagged = scaled_block<M>(blk, t, p == 0 ? 0 : 1, packed);
        store_tile<M>(tile, packed);
        if (flagged) record_tie(block, ties, tie_capacity, stats);
    }
}

// K7R: one selected block per thread into its window-local tile (region_tile_block); ties are recorded with the global
// block index, so exactly the blocks K7 (K7S) flags are flagged.  The selected blocks are one run per block row of
// each rectangle, so there is no box of consecutive blocks for one TMA load: the CTA's blocks come in by plain 16-byte
// loads of the pieces the arithmetic reads (block_pieces: 128 bytes at M = 8, 64 at M = 4, 16 at M = 2), consecutive
// threads on consecutive pieces, into K7's (K7S's) staging layout.
template <int M>
__global__ void __launch_bounds__(K7S_THREADS)
region_inverse_kernel(const int16_t* __restrict__ coef, hic_dct_geometry g, int n, RegionArgs a,
                      hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    constexpr int PIECES = block_pieces<M>();
    __shared__ int4 s_blk[K7S_THREADS * PIECES];
    __shared__ uint32_t s_src[K7S_THREADS];
    // 32-bit indices: the selected blocks are at most the batch's blocks, fewer than 2^32 (hic_dct_region and
    // hic_dct_scaled_region check it)
    const uint32_t nl = (uint32_t)a.s.ny_l * a.s.nx_l, nc = (uint32_t)a.s.ny_c * a.s.nx_c, per = nl + 2 * nc;
    const uint32_t first = blockIdx.x * K7S_THREADS, gid = first + threadIdx.x, total = per * (uint32_t)n;
    const bool live = gid < total;
    uint32_t img = 0;
    int p = 0, ly = 0, lx = 0;
    if (live) {
        img = gid / per;
        s_src[threadIdx.x] = (uint32_t)region_block<M>(g, a, img, gid - img * per, nl, nc, p, ly, lx);
    }
    __syncthreads();
    const int count = (int)min((uint32_t)K7S_THREADS, total - first);
    const int4* c4 = reinterpret_cast<const int4*>(coef);
    for (int q = threadIdx.x; q < PIECES * count; q += K7S_THREADS) {
        const int t = q / PIECES, j = q % PIECES;
        s_blk[staged_piece<M>(t, j)] = __ldg(c4 + (size_t)s_src[t] * 8 + j);
    }
    __syncthreads();
    if (!live) return;
    region_tile_block<M>(s_blk, threadIdx.x, p, region_tile<M>(a, img, p, ly, lx), s_src[threadIdx.x], ties, tie_capacity, stats);
}

// The fix-up of K7R's flagged blocks: inverse_fixup_kernel's arithmetic at M = 8, scaled_fixup_kernel's below, each
// block landing in its window-local tile.
template <int M>
__global__ void __launch_bounds__(128)
region_fixup_kernel(const int16_t* __restrict__ coef, hic_dct_geometry g, RegionArgs a,
                    const hic_tie_record* __restrict__ ties, uint32_t tie_capacity, uint32_t* __restrict__ stats) {
    auto tile = [&](const BlockPos& q) {
        const RegionFirst f = region_first<M>(g, a, q.img);
        if (q.p == 0) return region_tile<M>(a, q.img, 0, q.by - f.by_l, q.bx - f.bx_l);
        return region_tile<M>(a, q.img, q.p, q.by - f.by_c, q.bx - f.bx_c);
    };
    if constexpr (M == 8)
        inverse_fixup_body(coef, g, ties, tie_capacity, stats,
                           [&](int64_t img, int p, int by, int bx) { return BlockDst{tile({img, p, by, bx}), 8, 8, 0, 0}; });
    else
        scaled_fixup_body<M>(coef, g, ties, tie_capacity, stats, [&](uint32_t b) { return tile(block_pos(g, b)); });
}

// K8R: the colour stage over one window per image: a thread per chroma sample the window covers, producing the pixels
// of its 2x2 output quad that lie inside the window (cw = rw / 2 + 1 samples per row cover any origin's columns,
// ch = rh / 2 + 1 its rows).  The neighbours are chosen in the whole chroma planes with K8's borders (chroma_extent)
// and read from the window-local tiles; Y likewise; the n x rh x rw x 3 result is written directly.
template <int M>
__global__ void __launch_bounds__(256)
region_colour_kernel(hic_dct_geometry g, int n, RegionArgs a, uint8_t* __restrict__ rgb) {
    const int ch = a.rh / 2 + 1, cw = a.rw / 2 + 1;
    const int64_t per = (int64_t)ch * cw;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    const int top = __ldg(a.origin + 2 * img), left = __ldg(a.origin + 2 * img + 1);
    const int cy = (top >> 1) + (int)(rem / cw), cx = (left >> 1) + (int)(rem % cw);
    if (2 * cy > top + a.rh - 1 || 2 * cx > left + a.rw - 1) return;
    const RegionFirst f = region_first<M>(g, a, img);
    const int r0 = M * f.by_c, c0 = M * f.bx_c;
    const uint8_t* crp = a.cr + img * a.lc;
    const uint8_t* cbp = a.cb + img * a.lc;
    int up[2][4];
    chroma_up_quads(cy, cx, chroma_extent<M>(g), [&](int c, int r, int col) {
        return tile_sample<M>(c == 0 ? crp : cbp, a.s.nx_c, r - r0, col - c0);
    }, up);
    const uint8_t* ysrc = a.y + img * a.ly;
    uint8_t* dst = rgb + (size_t)img * a.rh * a.rw * 3;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const int oy = 2 * cy + dy, ox = 2 * cx + dx;
            if (oy < top || oy >= top + a.rh || ox < left || ox >= left + a.rw) continue;
            store_rgb(dst + ((size_t)(oy - top) * a.rw + (ox - left)) * 3,
                      tile_sample<M>(ysrc, a.s.nx_l, oy - M * f.by_l, ox - M * f.bx_l), up[0][2 * dy + dx], up[1][2 * dy + dx]);
        }
}
}  // namespace k7

// ------------------------------------------------------------------------------------------------
// layout converters
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
blocks_to_planes_kernel(const int16_t* __restrict__ coef, hic_dct_geometry g, int n, int32_t* __restrict__ lum,
                        int32_t* __restrict__ cr, int32_t* __restrict__ cb) {
    // one thread per coefficient, natural position inside the block varies fastest along x
    const int64_t per = g.blocks_per_image * 64;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    int64_t blk = rem >> 6;
    const int k = (int)(rem & 63);
    const int nat = c_zigzag[k];
    const int u = nat >> 3, v = nat & 7;
    int32_t* plane;
    int ph, pw, nbx;
    if (blk < g.nb_l) {
        plane = lum + (size_t)img * g.h * g.w; ph = g.h; pw = g.w; nbx = g.nbx_l;
    } else {
        blk -= g.nb_l;
        const int p = (int)(blk / g.nb_c);
        blk -= (int64_t)p * g.nb_c;
        plane = (p == 0 ? cr : cb) + (size_t)img * g.hc * g.wc; ph = g.hc; pw = g.wc; nbx = g.nbx_c;
    }
    const int y = 8 * (int)(blk / nbx) + u, x = 8 * (int)(blk % nbx) + v;
    if (y < ph && x < pw) plane[(size_t)y * pw + x] = (int32_t)coef[gid];
}

__global__ void __launch_bounds__(256)
planes_to_blocks_kernel(const int32_t* __restrict__ lum, const int32_t* __restrict__ cr,
                        const int32_t* __restrict__ cb, hic_dct_geometry g, int n, int16_t* __restrict__ coef) {
    const int64_t per = g.blocks_per_image * 64;
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid >= per * n) return;
    const int64_t img = gid / per;
    const int64_t rem = gid - img * per;
    int64_t blk = rem >> 6;
    const int k = (int)(rem & 63);
    const int nat = c_zigzag[k];
    const int u = nat >> 3, v = nat & 7;
    const int32_t* plane;
    int ph, pw, nbx;
    if (blk < g.nb_l) {
        plane = lum + (size_t)img * g.h * g.w; ph = g.h; pw = g.w; nbx = g.nbx_l;
    } else {
        blk -= g.nb_l;
        const int p = (int)(blk / g.nb_c);
        blk -= (int64_t)p * g.nb_c;
        plane = (p == 0 ? cr : cb) + (size_t)img * g.hc * g.wc; ph = g.hc; pw = g.wc; nbx = g.nbx_c;
    }
    const int y = 8 * (int)(blk / nbx) + u, x = 8 * (int)(blk % nbx) + v;
    coef[gid] = (y < ph && x < pw) ? (int16_t)plane[(size_t)y * pw + x] : (int16_t)0;
}

static inline unsigned grid_for(int64_t items, int threads) { return (unsigned)((items + threads - 1) / threads); }

// cuTensorMapEncodeTiled through the runtime (the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static int tensor_map_encoder(EncodeTiledFn* out) {
    static EncodeTiledFn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        HIC_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (qres != cudaDriverEntryPointSuccess || !fn) return hic::fail(HIC_ERR_CUDA, "cuTensorMapEncodeTiled is not available");
        encode = reinterpret_cast<EncodeTiledFn>(fn);
    }
    *out = encode;
    return HIC_OK;
}

// The decode entries' shared checks: n >= 1 images of h x w and (block_limit) a block count that fits 32-bit indices
static int batch_geometry(int32_t n, int32_t h, int32_t w, bool block_limit, hic_dct_geometry* g) {
    HIC_REQUIRE(n >= 1, "batch size must be positive");
    const int rc = geometry_of(h, w, g);
    if (rc) return rc;
    if (block_limit) HIC_REQUIRE((int64_t)n * g->blocks_per_image < (1ll << 32), "batch too large: %lld blocks", (long long)n * g->blocks_per_image);
    return HIC_OK;
}

// K7's [block][64 int16] view of the coefficient buffer; a box is the first box_cols entries of box_rows blocks
static int coef_block_map(CUtensorMap* map, const int16_t* d_coef, int64_t blocks, cuuint32_t box_cols, cuuint32_t box_rows,
                          CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2) {
    EncodeTiledFn encode = nullptr;
    const int rc = tensor_map_encoder(&encode);
    if (rc) return rc;
    const cuuint64_t dims[2] = {64, (cuuint64_t)blocks};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<int16_t*>(d_coef), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return hic::fail(HIC_ERR_CUDA, "cuTensorMapEncodeTiled (coefficient blocks) failed: %d", (int)r);
    return HIC_OK;
}

// f(std::integral_constant<int, M>()) for M = 8 / scale samples per block side: scale 2 or 4, or 1 too where FULL (the
// scaled launches leave it out, so that no scaled kernel is instantiated for M = 8)
template <bool FULL, class F>
static auto by_samples(int scale, F f) {
    if constexpr (FULL)
        if (scale == 1) return f(std::integral_constant<int, 8>());
    return scale == 2 ? f(std::integral_constant<int, 4>()) : f(std::integral_constant<int, 2>());
}

// K7S, its fix-up and K8S of hic_dct_scaled for M x M samples per block (scale 8 / M)
template <int M>
static int scaled_launch(const int16_t* d_coef, const hic_dct_geometry& g, int n, int sh, int sw, uint8_t* d_work,
                         hic_tie_record* d_ties, uint32_t tie_capacity, uint32_t* d_stats, uint8_t* d_rgb_out, cudaStream_t st) {
    const int64_t blocks = (int64_t)n * g.blocks_per_image;
    CUtensorMap tmap_blocks;
    const int rc = coef_block_map(&tmap_blocks, d_coef, blocks, M == 4 ? 32u : 8u, k7::K7S_THREADS,
                                  M == 4 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE);
    if (rc) return rc;
    const unsigned grid_inv = grid_for(blocks, k7::K7S_THREADS), grid_rgb = grid_for((int64_t)n * ((sh + 1) / 2) * ((sw + 1) / 2), 256);
    HIC_LAUNCH("scaled_inverse_kernel", st, k7::scaled_inverse_kernel<M><<<grid_inv, k7::K7S_THREADS, 0, st>>>(tmap_blocks, g, n, d_work, d_ties, tie_capacity, d_stats));
    HIC_LAUNCH("scaled_fixup_kernel", st, k7::scaled_fixup_kernel<M><<<148 * 4, 128, 0, st>>>(d_coef, g, d_work, d_ties, tie_capacity, d_stats));
    HIC_LAUNCH("scaled_colour_kernel", st, k7::scaled_colour_kernel<M><<<grid_rgb, 256, 0, st>>>(d_work, g, n, sh, sw, d_rgb_out));
    return HIC_OK;
}

// Every origin of the windowed entries names an rh x rw window inside the 1/scale image
static int check_origins(const hic_dct_geometry& g, int n, const int32_t* h_origin, int rh, int rw, int scale) {
    for (int i = 0; i < n; ++i) {
        const int rc = region_check(g, h_origin[2 * i], h_origin[2 * i + 1], rh, rw, scale);
        if (rc) return rc;
    }
    return HIC_OK;
}

// The body of hic_dct_region_blocks (scale 1) and hic_dct_scaled_region_blocks (scale 2 or 4)
static int region_blocks(int h, int w, int scale, int top, int left, int rh, int rw, int32_t* rect) {
    hic_dct_geometry g;
    int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    rc = region_check(g, top, left, rh, rw, scale);
    if (rc) return rc;
    by_samples<true>(scale, [&](auto m) { region_rect<decltype(m)::value>(g, top, left, rh, rw, rect); });
    return HIC_OK;
}

// The work buffer and tie capacity of n rh x rw windows at scale 1, 2 or 4, once the sizes entries' checks hold
static int region_sizes(int n, const hic_dct_geometry& g, int scale, int rh, int rw, size_t* work_bytes, uint32_t* tie_capacity) {
    const RegionLayout L = by_samples<true>(scale, [&](auto m) { return region_layout<decltype(m)::value>(n, g, rh, rw); });
    HIC_REQUIRE(L.blocks < (1ull << 32), "batch too large: %llu selected blocks", (unsigned long long)L.blocks);
    *work_bytes = L.total;
    *tie_capacity = (uint32_t)L.blocks;
    return HIC_OK;
}

// K7R, its fix-up and K8R of hic_dct_region (M = 8) and hic_dct_scaled_region (M = 4, 2) once the origins are
// checked; the origins are copied to the work buffer's head, the window-local tiles follow.  The launches keep the
// labels of the entry they serve: region_* at M = 8, scaled_region_* below.
template <int M>
static int region_launch(const int16_t* d_coef, const hic_dct_geometry& g, int n, const int32_t* h_origin, int rh, int rw,
                         uint8_t* d_work, size_t work_bytes, hic_tie_record* d_ties, uint32_t tie_capacity,
                         uint32_t* d_stats, uint8_t* d_rgb_out, cudaStream_t st) {
    constexpr bool full = M == 8;
    const RegionLayout L = region_layout<M>(n, g, rh, rw);
    HIC_REQUIRE(work_bytes >= L.total, "work buffer of %zu bytes is too small: %zu needed (%s)", work_bytes, L.total,
                full ? "hic_dct_region_sizes" : "hic_dct_scaled_region_sizes");
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_coef) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_work) & 15) == 0,
                "d_coef and d_work must be 16-byte aligned");
    const int rc = ensure_tables();
    if (rc) return rc;
    HIC_CUDA(cudaMemsetAsync(d_stats, 0, HIC_TIE_STATS * sizeof(uint32_t), st));
    HIC_CUDA(cudaMemcpyAsync(d_work, h_origin, (size_t)n * 2 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    uint8_t* y = d_work + L.head;     // the n images' Y tiles, then their Cr and their Cb tiles
    const k7::RegionArgs a = {reinterpret_cast<const int32_t*>(d_work), y, y + (size_t)n * L.ly, y + (size_t)n * (L.ly + L.lc),
                              L.ly, L.lc, L.s, rh, rw};
    HIC_LAUNCH(full ? "region_inverse_kernel" : "scaled_region_inverse_kernel", st, k7::region_inverse_kernel<M><<<grid_for((int64_t)L.blocks, k7::K7S_THREADS), k7::K7S_THREADS, 0, st>>>(d_coef, g, n, a, d_ties, tie_capacity, d_stats));
    HIC_LAUNCH(full ? "region_fixup_kernel" : "scaled_region_fixup_kernel", st, k7::region_fixup_kernel<M><<<148 * 4, 128, 0, st>>>(d_coef, g, a, d_ties, tie_capacity, d_stats));
    HIC_LAUNCH(full ? "region_colour_kernel" : "scaled_region_colour_kernel", st, k7::region_colour_kernel<M><<<grid_for((int64_t)n * (rh / 2 + 1) * (rw / 2 + 1), 256), 256, 0, st>>>(g, n, a, d_rgb_out));
    return HIC_OK;
}

}  // namespace hic

// ------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------
extern "C" {

int hic_dct_geometry_of(int32_t h, int32_t w, hic_dct_geometry* out) { return hic::geometry_of(h, w, out); }

int hic_dct_tie_capacity(int32_t n, int32_t h, int32_t w, uint32_t* out) {
    using namespace hic;
    HIC_REQUIRE(out != nullptr, "capacity output is NULL");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    hic_dct_geometry g;
    const int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    const int ext_x = max(8 * g.nbx_l, 16 * g.nbx_c), ext_y = max(8 * g.nby_l, 16 * g.nby_c);
    const uint64_t words = (uint64_t)ceil_div(ext_x, k1::TW) * ceil_div(ext_y, k1::TH) * n * k1::WARPS;
    const uint64_t cap = (uint64_t)n * g.blocks_per_image + (words * 4 + sizeof(hic_tie_record) - 1) / sizeof(hic_tie_record) + 1;
    HIC_REQUIRE(cap < (1ull << 32), "batch too large: %llu tie records", (unsigned long long)cap);
    *out = (uint32_t)cap;
    return HIC_OK;
}

int hic_dct_forward(const uint8_t* d_rgb, int32_t n, int32_t h, int32_t w, int16_t* d_coef, hic_tie_record* d_ties,
                    uint32_t tie_capacity, uint32_t* d_stats, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_rgb && d_coef && d_ties && d_stats, "NULL device pointer");
    HIC_REQUIRE(n >= 1 && n <= 65535, "batch size must be in 1..65535 (got %d)", n);
    hic_dct_geometry g;
    int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    HIC_REQUIRE((int64_t)n * g.blocks_per_image < (1ll << 32), "batch too large: %lld blocks", (long long)n * g.blocks_per_image);
    rc = ensure_tables();
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    HIC_CUDA(cudaMemsetAsync(d_stats, 0, HIC_TIE_STATS * sizeof(uint32_t), st));
    const int ext_x = max(8 * g.nbx_l, 16 * g.nbx_c), ext_y = max(8 * g.nby_l, 16 * g.nby_c);
    dim3 grid(ceil_div(ext_x, k1::TW), ceil_div(ext_y, k1::TH), n);
    // the flag words of K1 (one per warp) live at the tail of the tie buffer, the list of flagged blocks at its head
    const uint64_t flag_words64 = (uint64_t)grid.x * grid.y * grid.z * k1::WARPS;
    HIC_REQUIRE(flag_words64 < (1ull << 32), "batch too large: %llu tiles", (unsigned long long)(flag_words64 / k1::WARPS));
    const uint32_t flag_words = (uint32_t)flag_words64, flag_slots = (flag_words * 4u + (uint32_t)sizeof(hic_tie_record) - 1u) / (uint32_t)sizeof(hic_tie_record);
    if (tie_capacity <= flag_slots)
        return hic::fail(HIC_ERR_CAPACITY, "tie_capacity %u is too small: the flag words alone take %u records (hic_dct_tie_capacity)", tie_capacity, flag_slots);
    const uint32_t list_capacity = tie_capacity - flag_slots;
    uint32_t* flagmap = reinterpret_cast<uint32_t*>(d_ties + list_capacity);
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_coef) & 127) == 0, "d_coef must be 128-byte aligned");
    static bool attr_set[64] = {false};
    int dev = 0;
    HIC_CUDA(cudaGetDevice(&dev));
    if (dev >= 64 || !attr_set[dev]) {
        HIC_CUDA(cudaFuncSetAttribute(k1::forward_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(k1::Smem)));
        HIC_CUDA(cudaFuncSetAttribute(k1::forward_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(k1::Smem)));
        if (dev < 64) attr_set[dev] = true;
    }
    EncodeTiledFn encode = nullptr;
    rc = tensor_map_encoder(&encode);
    if (rc) return rc;
    const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    // TMA load: the image batch as a 3-D tensor of 32-bit words (3W/4 words, H rows, n images)
    CUtensorMap tmap, tmap_rows;
    memset(&tmap, 0, sizeof(tmap));
    memset(&tmap_rows, 0, sizeof(tmap_rows));
    bool use_tma = (w % 16 == 0) && ((reinterpret_cast<uintptr_t>(d_rgb) & 15) == 0) && getenv("HIC_NO_TMA") == nullptr;
    if (use_tma) {
        const cuuint64_t dims[3] = {(cuuint64_t)w * 3 / 4, (cuuint64_t)h, (cuuint64_t)n};
        const cuuint64_t strides[2] = {(cuuint64_t)w * 3, (cuuint64_t)w * 3 * h};
        const cuuint32_t box[3] = {(cuuint32_t)k1::RWORDS, (cuuint32_t)k1::RH, 1};
        const CUresult r = encode(&tmap, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(d_rgb), dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        const cuuint32_t box_rows[3] = {(cuuint32_t)k1::RWORDS, (cuuint32_t)k1::CHUNK_ROWS, 1};
        const CUresult r2 = encode(&tmap_rows, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t*>(d_rgb), dims, strides, box_rows, estr,
                                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS || r2 != CUDA_SUCCESS) use_tma = false;       // fall back to the generic loader
        if (getenv("HIC_DEBUG")) fprintf(stderr, "[hic] tensor map encode -> %d (use_tma=%d)\n", (int)r, (int)use_tma);
    }
    // TMA stores: the coefficient buffer as [image][block row][block column][64 int16] (luminance) and
    // [image][plane][block row][block column][64 int16] (Cr, Cb), one 128-byte block = one swizzle row
    CUtensorMap tmap_l, tmap_c;
    {
        const cuuint64_t blk = 128, img_stride = blk * (cuuint64_t)g.blocks_per_image;
        const cuuint64_t dims_l[4] = {64, (cuuint64_t)g.nbx_l, (cuuint64_t)g.nby_l, (cuuint64_t)n};
        const cuuint64_t str_l[3] = {blk, blk * (cuuint64_t)g.nbx_l, img_stride};
        const cuuint32_t box_l[4] = {64, k1::TW / 8, k1::TH / 8, 1};
        CUresult r = encode(&tmap_l, CU_TENSOR_MAP_DATA_TYPE_UINT16, 4, d_coef, dims_l, str_l, box_l, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return hic::fail(HIC_ERR_CUDA, "cuTensorMapEncodeTiled (luminance blocks) failed: %d", (int)r);
        const cuuint64_t dims_c[5] = {64, (cuuint64_t)g.nbx_c, (cuuint64_t)g.nby_c, 2, (cuuint64_t)n};
        const cuuint64_t str_c[4] = {blk, blk * (cuuint64_t)g.nbx_c, blk * (cuuint64_t)g.nb_c, img_stride};
        const cuuint32_t box_c[5] = {64, k1::CW / 8, k1::CH / 8, 2, 1};
        r = encode(&tmap_c, CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, d_coef + (size_t)g.nb_l * 64, dims_c, str_c, box_c, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return hic::fail(HIC_ERR_CUDA, "cuTensorMapEncodeTiled (chroma blocks) failed: %d", (int)r);
    }
    if (use_tma)
        HIC_LAUNCH("forward_kernel", st, k1::forward_kernel<true><<<grid, k1::THREADS, sizeof(k1::Smem), st>>>(tmap, tmap_rows, tmap_l, tmap_c, d_rgb, h, w, g, flagmap));
    else
        HIC_LAUNCH("forward_kernel", st, k1::forward_kernel<false><<<grid, k1::THREADS, sizeof(k1::Smem), st>>>(tmap, tmap_rows, tmap_l, tmap_c, d_rgb, h, w, g, flagmap));
    HIC_LAUNCH("tie_list_kernel", st, k1::tie_list_kernel<<<min(148u * 8u, (flag_words + 255u) / 256u), 256, 0, st>>>(flagmap, flag_words, (int)grid.x, (int)grid.y, g, h, w, d_ties, list_capacity, d_stats));
    HIC_LAUNCH("fixup_kernel", st, k1::fixup_kernel<<<148 * 8, 32 * k1::FIX_WARPS, 0, st>>>(d_rgb, h, w, g, d_coef, d_ties, list_capacity, d_stats));
    return HIC_OK;
}

int hic_blocks_to_planes(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t* d_lum, int32_t* d_cr,
                         int32_t* d_cb, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && d_lum && d_cr && d_cb, "NULL device pointer");
    hic_dct_geometry g;
    const int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    const int64_t items = (int64_t)n * g.blocks_per_image * 64;
    cudaStream_t st = as_stream(stream);
    HIC_LAUNCH("blocks_to_planes_kernel", st, blocks_to_planes_kernel<<<grid_for(items, 256), 256, 0, st>>>(d_coef, g, n, d_lum, d_cr, d_cb));
    return HIC_OK;
}

int hic_planes_to_blocks(const int32_t* d_lum, const int32_t* d_cr, const int32_t* d_cb, int32_t n, int32_t h,
                         int32_t w, int16_t* d_coef, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && d_lum && d_cr && d_cb, "NULL device pointer");
    hic_dct_geometry g;
    const int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    const int64_t items = (int64_t)n * g.blocks_per_image * 64;
    cudaStream_t st = as_stream(stream);
    HIC_LAUNCH("planes_to_blocks_kernel", st, planes_to_blocks_kernel<<<grid_for(items, 256), 256, 0, st>>>(d_lum, d_cr, d_cb, g, n, d_coef));
    return HIC_OK;
}

int hic_dct_inverse(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, uint8_t* d_y, uint8_t* d_cr,
                    uint8_t* d_cb, uint8_t* d_rgb_out, hic_tie_record* d_ties, uint32_t tie_capacity,
                    uint32_t* d_stats, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && d_y && d_cr && d_cb && d_rgb_out && d_ties && d_stats, "NULL device pointer");
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, true, &g);
    if (rc) return rc;
    rc = ensure_tables();
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    HIC_CUDA(cudaMemsetAsync(d_stats, 0, HIC_TIE_STATS * sizeof(uint32_t), st));
    const int64_t blocks = (int64_t)n * g.blocks_per_image;
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_coef) & 127) == 0, "d_coef must be 128-byte aligned");
    CUtensorMap tmap_blocks;
    rc = coef_block_map(&tmap_blocks, d_coef, blocks, 64, k7::K7_THREADS, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
    if (rc) return rc;
    HIC_LAUNCH("inverse_kernel", st, k7::inverse_kernel<<<grid_for(blocks, k7::K7_THREADS), k7::K7_THREADS, 0, st>>>(tmap_blocks, g, n, d_y, d_cr, d_cb, d_ties, tie_capacity, d_stats));
    HIC_LAUNCH("inverse_fixup_kernel", st, k7::inverse_fixup_kernel<<<148 * 4, 128, 0, st>>>(d_coef, g, d_y, d_cr, d_cb, d_ties, tie_capacity, d_stats));
    const int64_t quads = (int64_t)n * g.hc * g.wc;
    const bool word_rows = g.wc % 4 == 0 && g.w % 8 == 0 && ((g.h * (int64_t)g.w) % 8 == 0) && ((g.hc * (int64_t)g.wc) % 4 == 0) &&
                           ((reinterpret_cast<uintptr_t>(d_y) & 7) == 0) && ((reinterpret_cast<uintptr_t>(d_cr) & 3) == 0) &&
                           ((reinterpret_cast<uintptr_t>(d_cb) & 3) == 0) && ((reinterpret_cast<uintptr_t>(d_rgb_out) & 3) == 0);
    if (word_rows)
        HIC_LAUNCH("upsample_colour_kernel", st, k7::upsample_colour_vec_kernel<<<grid_for(quads / 4, 256), 256, 0, st>>>(d_y, d_cr, d_cb, g, n, d_rgb_out));
    else
        HIC_LAUNCH("upsample_colour_kernel", st, k7::upsample_colour_kernel<<<grid_for(quads, 256), 256, 0, st>>>(d_y, d_cr, d_cb, g, n, d_rgb_out));
    return HIC_OK;
}

int hic_dct_thumbnail_shape(int32_t h, int32_t w, int32_t* th, int32_t* tw) {
    using namespace hic;
    HIC_REQUIRE(th && tw, "NULL argument");
    hic_dct_geometry g;
    const int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    *th = ceil_div(g.out_h, 8);
    *tw = ceil_div(g.out_w, 8);
    return HIC_OK;
}

int hic_dct_thumbnail(const int16_t* d_dc, int32_t n, int32_t h, int32_t w, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_dc && d_rgb_out, "NULL device pointer");
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    int32_t th = 0, tw = 0;
    rc = hic_dct_thumbnail_shape(h, w, &th, &tw);
    if (rc) return rc;
    rc = ensure_tables();
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    HIC_LAUNCH("thumbnail_kernel", st, k7::thumbnail_kernel<<<grid_for((int64_t)n * th * tw, 256), 256, 0, st>>>(d_dc, g, n, th, tw, d_rgb_out));
    return HIC_OK;
}

int hic_dct_region_blocks(int32_t h, int32_t w, int32_t top, int32_t left, int32_t rh, int32_t rw, int32_t* rect) {
    using namespace hic;
    HIC_REQUIRE(rect != nullptr, "NULL argument");
    return region_blocks(h, w, 1, top, left, rh, rw, rect);
}

int hic_dct_region_sizes(int32_t n, int32_t h, int32_t w, int32_t rh, int32_t rw, size_t* work_bytes, uint32_t* tie_capacity) {
    using namespace hic;
    HIC_REQUIRE(work_bytes && tie_capacity, "NULL argument");
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    rc = region_check(g, 0, 0, rh, rw);
    if (rc) return rc;
    return region_sizes(n, g, 1, rh, rw, work_bytes, tie_capacity);
}

int hic_dct_region(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, const int32_t* h_origin, int32_t rh,
                   int32_t rw, uint8_t* d_work, size_t work_bytes, hic_tie_record* d_ties, uint32_t tie_capacity,
                   uint32_t* d_stats, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && h_origin && d_work && d_ties && d_stats && d_rgb_out, "NULL pointer");
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, true, &g);
    if (rc) return rc;
    rc = check_origins(g, n, h_origin, rh, rw, 1);
    if (rc) return rc;
    return region_launch<8>(d_coef, g, n, h_origin, rh, rw, d_work, work_bytes, d_ties, tie_capacity, d_stats, d_rgb_out,
                            as_stream(stream));
}

int hic_dct_scaled_shape(int32_t h, int32_t w, int32_t scale, int32_t* sh, int32_t* sw) {
    using namespace hic;
    HIC_REQUIRE(sh && sw, "NULL argument");
    HIC_REQUIRE(scale == 2 || scale == 4, "scale must be 2 or 4 (got %d; scale 8 is hic_dct_thumbnail)", scale);
    hic_dct_geometry g;
    const int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    *sh = ceil_div(g.out_h, scale);
    *sw = ceil_div(g.out_w, scale);
    return HIC_OK;
}

int hic_dct_scaled_sizes(int32_t n, int32_t h, int32_t w, int32_t scale, size_t* work_bytes, uint32_t* tie_capacity) {
    using namespace hic;
    HIC_REQUIRE(work_bytes && tie_capacity, "NULL argument");
    HIC_REQUIRE(n >= 1, "batch size must be positive");
    HIC_REQUIRE(scale == 2 || scale == 4, "scale must be 2 or 4 (got %d; scale 8 is hic_dct_thumbnail)", scale);
    hic_dct_geometry g;
    const int rc = geometry_of(h, w, &g);
    if (rc) return rc;
    const int64_t blocks = (int64_t)n * g.blocks_per_image;
    HIC_REQUIRE(blocks < (1ll << 32), "batch too large: %lld blocks", (long long)blocks);
    const int m = 8 / scale;
    *work_bytes = (size_t)blocks * m * m;
    *tie_capacity = (uint32_t)blocks;
    return HIC_OK;
}

int hic_dct_scaled(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t scale, uint8_t* d_work, size_t work_bytes,
                   hic_tie_record* d_ties, uint32_t tie_capacity, uint32_t* d_stats, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && d_work && d_ties && d_stats && d_rgb_out, "NULL device pointer");
    size_t need = 0;
    uint32_t cap = 0;
    int rc = hic_dct_scaled_sizes(n, h, w, scale, &need, &cap);
    if (rc) return rc;
    HIC_REQUIRE(work_bytes >= need, "work buffer of %zu bytes is too small: %zu needed (hic_dct_scaled_sizes)", work_bytes, need);
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_coef) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_work) & 15) == 0,
                "d_coef and d_work must be 16-byte aligned");
    hic_dct_geometry g;           // what hic_dct_scaled_sizes checked
    rc = geometry_of(h, w, &g);
    if (rc) return rc;
    const int sh = ceil_div(g.out_h, scale), sw = ceil_div(g.out_w, scale);
    rc = ensure_tables();
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    HIC_CUDA(cudaMemsetAsync(d_stats, 0, HIC_TIE_STATS * sizeof(uint32_t), st));
    return by_samples<false>(scale, [&](auto m) {
        return scaled_launch<decltype(m)::value>(d_coef, g, n, sh, sw, d_work, d_ties, tie_capacity, d_stats, d_rgb_out, st);
    });
}

int hic_dct_scaled_region_blocks(int32_t h, int32_t w, int32_t scale, int32_t top, int32_t left, int32_t rh, int32_t rw,
                                 int32_t* rect) {
    using namespace hic;
    HIC_REQUIRE(rect != nullptr, "NULL argument");
    HIC_REQUIRE(scale == 2 || scale == 4, "scale must be 2 or 4 (got %d)", scale);
    return region_blocks(h, w, scale, top, left, rh, rw, rect);
}

int hic_dct_scaled_region_sizes(int32_t n, int32_t h, int32_t w, int32_t scale, int32_t rh, int32_t rw, size_t* work_bytes,
                                uint32_t* tie_capacity) {
    using namespace hic;
    HIC_REQUIRE(work_bytes && tie_capacity, "NULL argument");
    HIC_REQUIRE(scale == 2 || scale == 4 || scale == 8, "scale must be 2, 4 or 8 (got %d)", scale);
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    rc = region_check(g, 0, 0, rh, rw, scale);
    if (rc) return rc;
    if (scale == 8) {              // hic_dct_thumbnail_region: the origins alone, no tie stage
        *work_bytes = (size_t)n * 2 * sizeof(int32_t);
        *tie_capacity = 0;
        return HIC_OK;
    }
    return region_sizes(n, g, scale, rh, rw, work_bytes, tie_capacity);
}

int hic_dct_scaled_region(const int16_t* d_coef, int32_t n, int32_t h, int32_t w, int32_t scale, const int32_t* h_origin,
                          int32_t rh, int32_t rw, uint8_t* d_work, size_t work_bytes, hic_tie_record* d_ties,
                          uint32_t tie_capacity, uint32_t* d_stats, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_coef && h_origin && d_work && d_ties && d_stats && d_rgb_out, "NULL pointer");
    HIC_REQUIRE(scale == 2 || scale == 4, "scale must be 2 or 4 (got %d; the 1/8-scale window is hic_dct_thumbnail_region)", scale);
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, true, &g);
    if (rc) return rc;
    rc = check_origins(g, n, h_origin, rh, rw, scale);
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    return by_samples<false>(scale, [&](auto m) {
        return region_launch<decltype(m)::value>(d_coef, g, n, h_origin, rh, rw, d_work, work_bytes, d_ties, tie_capacity,
                                                 d_stats, d_rgb_out, st);
    });
}

int hic_dct_thumbnail_region(const int16_t* d_dc, int32_t n, int32_t h, int32_t w, const int32_t* h_origin, int32_t rh,
                             int32_t rw, uint8_t* d_work, size_t work_bytes, uint8_t* d_rgb_out, void* stream) {
    using namespace hic;
    HIC_REQUIRE(d_dc && h_origin && d_work && d_rgb_out, "NULL pointer");
    hic_dct_geometry g;
    int rc = batch_geometry(n, h, w, false, &g);
    if (rc) return rc;
    rc = check_origins(g, n, h_origin, rh, rw, 8);
    if (rc) return rc;
    const size_t need = (size_t)n * 2 * sizeof(int32_t);
    HIC_REQUIRE(work_bytes >= need, "work buffer of %zu bytes is too small: %zu needed (hic_dct_scaled_region_sizes)", work_bytes, need);
    HIC_REQUIRE((reinterpret_cast<uintptr_t>(d_dc) & 1) == 0 && (reinterpret_cast<uintptr_t>(d_work) & 3) == 0,
                "d_dc must be 2-byte aligned and d_work 4-byte aligned");
    rc = ensure_tables();
    if (rc) return rc;
    cudaStream_t st = as_stream(stream);
    HIC_CUDA(cudaMemcpyAsync(d_work, h_origin, need, cudaMemcpyHostToDevice, st));
    HIC_LAUNCH("thumbnail_region_kernel", st, k7::thumbnail_region_kernel<<<grid_for((int64_t)n * rh * rw, 256), 256, 0, st>>>(d_dc, g, n, reinterpret_cast<const int32_t*>(d_work), rh, rw, d_rgb_out));
    return HIC_OK;
}

}  // extern "C"
