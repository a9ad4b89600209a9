// hic_core.cuh -- arithmetic shared by the sm_100a kernels and the host-side check harness.
//
// Everything here is `__host__ __device__` so that the exact same arithmetic the kernels run can be
// exercised on the CPU (tests/cpu_harness) before any GPU time is spent.  Reference citations are
// into /root/reference (nhomble/hiccup).
#pragma once
#include <stdint.h>
#include <math.h>

#ifdef __CUDACC__
#define HIC_HD __host__ __device__ __forceinline__
#else
#define HIC_HD inline
#endif

namespace hic {

// ------------------------------------------------------------------------------------------------
// constants
// ------------------------------------------------------------------------------------------------
// Annex-K tables, natural (row-major) order -- reference hiccup/quantization.py:14-37.
#define HIC_LUM_TABLE { \
    16, 11, 10, 16, 24, 40, 51, 61,   12, 12, 14, 19, 26, 58, 60, 55, \
    14, 13, 16, 24, 40, 57, 69, 56,   14, 17, 22, 29, 51, 87, 80, 62, \
    18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113, 92, \
    49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99 }
#define HIC_CHROMA_TABLE { \
    17, 18, 24, 47, 99, 99, 99, 99,   18, 21, 26, 66, 99, 99, 99, 99, \
    24, 26, 56, 99, 99, 99, 99, 99,   47, 66, 99, 99, 99, 99, 99, 99, \
    99, 99, 99, 99, 99, 99, 99, 99,   99, 99, 99, 99, 99, 99, 99, 99, \
    99, 99, 99, 99, 99, 99, 99, 99,   99, 99, 99, 99, 99, 99, 99, 99 }

// Scan order of reference transform._zigzag_indices (transform.py:106-124): anti-diagonals d = x+y,
// even d with y ascending, odd d with y descending (the transpose of the standard JPEG scan).
// Entry k is the natural index 8*y + x read at scan position k.
#define HIC_ZIGZAG8 { \
    0, 8, 1, 2, 9, 16, 24, 17, 10, 3, 4, 11, 18, 25, 32, 40, 33, 26, 19, 12, 5, 6, 13, 20, 27, 34, 41, 48, \
    56, 49, 42, 35, 28, 21, 14, 7, 15, 22, 29, 36, 43, 50, 57, 58, 51, 44, 37, 30, 23, 31, 38, 45, 52, \
    59, 60, 53, 46, 39, 47, 54, 61, 62, 55, 63 }

// ------------------------------------------------------------------------------------------------
// float64 helpers that are never contracted into FMAs (the reference's scipy/numpy builds are
// plain x86-64: separate multiply and add, each rounded).  Host builds use -ffp-contract=off.
// ------------------------------------------------------------------------------------------------
HIC_HD double dmul(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
HIC_HD double dadd(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}
HIC_HD double dsub(double a, double b) {
#ifdef __CUDA_ARCH__
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}
HIC_HD double ddiv(double a, double b) {
#ifdef __CUDA_ARCH__
    return __ddiv_rn(a, b);
#else
    return a / b;
#endif
}

// ------------------------------------------------------------------------------------------------
// scipy.fftpack.dct / idct (ducc0) for N = 8, operation for operation in float64.
//
// ducc0 T_dcst23<double>::exec: type 2 = pre-butterflies, backward real FFT of length 8 run as a
// radix-2 pass (l1=1, ido=4) then a radix-4 pass (l1=2, ido=1), post-twiddle; type 3 = the mirror.
// Twiddles are ducc0's UnityRoots<double> values (two small tables multiplied in double), which
// differ from correctly rounded cosines by an ulp; they are embedded as hex literals and checked
// against the oracle's run-time derivation in tests/test_oracle_dct.py.
// Reference call sites: hiccup/transform.py:80,82 (dct2) and :99,101 (idct2).
// ------------------------------------------------------------------------------------------------
#define HIC_TW0 0x1.f6297cff75cb0p-1   /* cos(1*pi/16) */
#define HIC_TW1 0x1.d906bcf328d46p-1   /* cos(2*pi/16) */
#define HIC_TW2 0x1.a9b66290ea1a3p-1   /* cos(3*pi/16) */
#define HIC_TW3 0x1.6a09e667f3bccp-1   /* cos(4*pi/16), one ulp below the rounded value */
#define HIC_TW4 0x1.1c73b39ae68c8p-1   /* cos(5*pi/16) */
#define HIC_TW5 0x1.87de2a6aea963p-2   /* cos(6*pi/16) */
#define HIC_TW6 0x1.8f8b83c69a60ap-3   /* cos(7*pi/16) */
#define HIC_WR  0x1.6a09e667f3bccp-1   /* Re exp(2 pi i / 8) */
#define HIC_WI  0x1.6a09e667f3bcdp-1   /* Im exp(2 pi i / 8) */

HIC_HD void ducc_dct2_8(double* c) {
    const double c0 = dmul(c[0], 2.0), c7 = dmul(c[7], 2.0);
    const double c2 = dsub(c[2], c[1]), c1 = dadd(c[2], c[1]);
    const double c4 = dsub(c[4], c[3]), c3 = dadd(c[4], c[3]);
    const double c6 = dsub(c[6], c[5]), c5 = dadd(c[6], c[5]);
    // radix-2 backward pass
    double a[8];
    a[0] = dadd(c0, c7);
    a[4] = dsub(c0, c7);
    a[3] = dmul(2.0, c3);
    a[7] = dmul(-2.0, c4);
    a[1] = dadd(c1, c5);
    const double tr2 = dsub(c1, c5);
    const double ti2 = dadd(c2, c6);
    a[2] = dsub(c2, c6);
    a[6] = dadd(dmul(HIC_WR, ti2), dmul(HIC_WI, tr2));
    a[5] = dsub(dmul(HIC_WR, tr2), dmul(HIC_WI, ti2));
    // radix-4 backward pass
    double r[8];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double t2 = dadd(a[4 * k], a[4 * k + 3]);
        const double t1 = dsub(a[4 * k], a[4 * k + 3]);
        const double t3 = dmul(2.0, a[4 * k + 1]);
        const double t4 = dmul(2.0, a[4 * k + 2]);
        r[k] = dadd(t2, t3);
        r[k + 4] = dsub(t2, t3);
        r[k + 6] = dadd(t1, t4);
        r[k + 2] = dsub(t1, t4);
    }
    c[0] = r[0];
    {
        const double t1 = dadd(dmul(HIC_TW0, r[7]), dmul(HIC_TW6, r[1]));
        const double t2 = dsub(dmul(HIC_TW0, r[1]), dmul(HIC_TW6, r[7]));
        c[1] = dmul(0.5, dadd(t1, t2));
        c[7] = dmul(0.5, dsub(t1, t2));
    }
    {
        const double t1 = dadd(dmul(HIC_TW1, r[6]), dmul(HIC_TW5, r[2]));
        const double t2 = dsub(dmul(HIC_TW1, r[2]), dmul(HIC_TW5, r[6]));
        c[2] = dmul(0.5, dadd(t1, t2));
        c[6] = dmul(0.5, dsub(t1, t2));
    }
    {
        const double t1 = dadd(dmul(HIC_TW2, r[5]), dmul(HIC_TW4, r[3]));
        const double t2 = dsub(dmul(HIC_TW2, r[3]), dmul(HIC_TW4, r[5]));
        c[3] = dmul(0.5, dadd(t1, t2));
        c[5] = dmul(0.5, dsub(t1, t2));
    }
    c[4] = dmul(r[4], HIC_TW3);
}

HIC_HD void ducc_dct3_8(double* c) {
    {
        const double t1 = dadd(c[1], c[7]), t2 = dsub(c[1], c[7]);
        c[1] = dadd(dmul(HIC_TW0, t2), dmul(HIC_TW6, t1));
        c[7] = dsub(dmul(HIC_TW0, t1), dmul(HIC_TW6, t2));
    }
    {
        const double t1 = dadd(c[2], c[6]), t2 = dsub(c[2], c[6]);
        c[2] = dadd(dmul(HIC_TW1, t2), dmul(HIC_TW5, t1));
        c[6] = dsub(dmul(HIC_TW1, t1), dmul(HIC_TW5, t2));
    }
    {
        const double t1 = dadd(c[3], c[5]), t2 = dsub(c[3], c[5]);
        c[3] = dadd(dmul(HIC_TW2, t2), dmul(HIC_TW4, t1));
        c[5] = dsub(dmul(HIC_TW2, t1), dmul(HIC_TW4, t2));
    }
    c[4] = dmul(c[4], dmul(2.0, HIC_TW3));
    // radix-4 forward pass (l1=2, ido=1)
    double h[8];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
        const double p0 = c[k], p1 = c[k + 2], p2 = c[k + 4], p3 = c[k + 6];
        const double tr1 = dadd(p3, p1);
        h[2 + 4 * k] = dsub(p3, p1);
        const double tr2 = dadd(p0, p2);
        h[1 + 4 * k] = dsub(p0, p2);
        h[0 + 4 * k] = dadd(tr2, tr1);
        h[3 + 4 * k] = dsub(tr2, tr1);
    }
    // radix-2 forward pass (l1=1, ido=4)
    double r[8];
    r[0] = dadd(h[0], h[4]);
    r[7] = dsub(h[0], h[4]);
    r[4] = -h[7];
    r[3] = h[3];
    const double tr2 = dadd(dmul(HIC_WR, h[5]), dmul(HIC_WI, h[6]));
    const double ti2 = dsub(dmul(HIC_WR, h[6]), dmul(HIC_WI, h[5]));
    r[1] = dadd(h[1], tr2);
    r[5] = dsub(h[1], tr2);
    r[2] = dadd(ti2, h[2]);
    r[6] = dsub(ti2, h[2]);
    c[0] = r[0];
    c[7] = r[7];
    c[1] = dsub(r[1], r[2]);
    c[2] = dadd(r[1], r[2]);
    c[3] = dsub(r[3], r[4]);
    c[4] = dadd(r[3], r[4]);
    c[5] = dsub(r[5], r[6]);
    c[6] = dadd(r[5], r[6]);
}

// round half to even, as np.round (reference quantization.py:80-81)
HIC_HD int32_t round_half_even(double v) {
#ifdef __CUDA_ARCH__
    return __double2int_rn(v);
#else
    return (int32_t)nearbyint(v);
#endif
}

// One quantised coefficient exactly as the reference computes it: rows then columns through
// ducc0's DCT (transform.py:67-84), true division by the table entry, np.round, int32.
// px: the 8x8 block after the -128 shift and zero padding, row major.  (u, v) = (row, col).
HIC_HD int32_t exact_quantised_coef(const int16_t* px, int u, int v, int q) {
    double col[8];
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
        double row[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) row[j] = (double)px[8 * i + j];
        ducc_dct2_8(row);
        col[i] = row[v];
    }
    ducc_dct2_8(col);
    return round_half_even(ddiv(col[u], (double)q));
}

// The whole quantised block exactly as the reference computes it (16 eight-point transforms).
// px: x - 128, zero padded, row major; q: the table, row major; out: natural order.
HIC_HD void exact_quantised_block(const int16_t* px, const int* q, int32_t* out) {
    double a[64];
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
        double row[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) row[j] = (double)px[8 * i + j];
        ducc_dct2_8(row);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[8 * i + j] = row[j];
    }
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        double col[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) col[i] = a[8 * i + j];
        ducc_dct2_8(col);
#pragma unroll
        for (int i = 0; i < 8; ++i) out[8 * i + j] = round_half_even(ddiv(col[i], (double)q[8 * i + j]));
    }
}

// The whole decoded block exactly as the reference computes it.  cq: coef * table, natural order;
// out: the float64 samples before the uint8 cast, row major.
HIC_HD void exact_decoded_block(const int32_t* cq, double* out) {
    double a[64];
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
        double row[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) row[j] = (double)cq[8 * i + j];
        ducc_dct3_8(row);
#pragma unroll
        for (int j = 0; j < 8; ++j) a[8 * i + j] = row[j];
    }
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        double col[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) col[i] = a[8 * i + j];
        ducc_dct3_8(col);
#pragma unroll
        for (int i = 0; i < 8; ++i) out[8 * i + j] = dadd(ddiv(col[i], 256.0), 128.0);
    }
}

// One decoded sample exactly as the reference computes it (transform.py:169-179, 87-103):
// coef*table, idct rows then columns, /256, +128, astype(uint8) = truncate toward zero, wrap.
// cq: the dequantised 8x8 block (coef * table), row major.  Returns the float64 value before the
// uint8 cast so callers can count near-integer cases.
HIC_HD double exact_decoded_sample(const int32_t* cq, int y, int x) {
    double col[8];
#pragma unroll 1
    for (int i = 0; i < 8; ++i) {
        double row[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) row[j] = (double)cq[8 * i + j];
        ducc_dct3_8(row);
        col[i] = row[x];
    }
    ducc_dct3_8(col);
    return dadd(ddiv(col[y], 256.0), 128.0);
}

HIC_HD uint8_t wrap_u8(double v) {            // numpy float64 -> uint8 cast on x86-64
    return (uint8_t)((long long)v & 0xFF);    // (long long) truncates toward zero
}

// ------------------------------------------------------------------------------------------------
// colour conversion: OpenCV's 14-bit fixed point (reference compression.py:21,56)
// ------------------------------------------------------------------------------------------------
HIC_HD void rgb_to_ycrcb(int r, int g, int b, int& y, int& cr, int& cb) {
    y = (4899 * r + 9617 * g + 1868 * b + 8192) >> 14;
    cr = ((r - y) * 11682 + (128 << 14) + 8192) >> 14;
    cb = ((b - y) * 9241 + (128 << 14) + 8192) >> 14;
    cr = cr < 0 ? 0 : (cr > 255 ? 255 : cr);
    cb = cb < 0 ? 0 : (cb > 255 ? 255 : cb);
}

HIC_HD int clamp_u8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

HIC_HD void ycrcb_to_rgb(int y, int cr, int cb, int& r, int& g, int& b) {
    cr -= 128;
    cb -= 128;
    r = clamp_u8(y + ((cr * 22987 + 8192) >> 14));
    g = clamp_u8(y + ((cb * -5636 + cr * -11698 + 8192) >> 14));
    b = clamp_u8(y + ((cb * 29049 + 8192) >> 14));
}

// BORDER_REFLECT_101 index, then clamped (tiles may overhang far past a small image; those
// positions are masked out downstream, the clamp only keeps the address legal)
HIC_HD int reflect101(int i, int n) {
    if (i < 0) i = -i;
    if (i >= n) i = 2 * n - 2 - i;
    return i < 0 ? 0 : (i >= n ? n - 1 : i);
}

// ------------------------------------------------------------------------------------------------
// fast float32 8-point transforms: even / odd split with a DENSE odd part.
//
// Forward (DCT-II): s_i = x_i + x_{7-i}, d_i = x_i - x_{7-i}; the even outputs are a 4-point DCT of s
// (two butterflies + one rotation written as two FMAs), the odd outputs are the 4x4 matrix
// cos((2i+1) k pi / 16) applied to d with every row divided by its first entry, i.e. three FMAs per
// output.  8 + 8 + 12 = 28 operations (Arai-Agui-Nakajima needs 29 adds + 5 multiplies: it saves
// multiplications, which cost nothing on FMA hardware), and -- what matters here -- no cancellation between
// large intermediates: a rigorous first-order bound of the float32 rounding error of the two-pass 8x8
// transform is 12.6 units of 4 u E (u = 2^-24, E = sum |x|) for the worst coefficient against 224 for AAN,
// and 9.8 units of 4 u S / 256 against 337 for the inverse (csrc/hic_dct_bound.h derives the bounds from
// THIS code by running it on a value type that carries error bounds; tools/dct_error_bound.py is the
// independent Python derivation; tests/test_oracle_dct.py compares the two and searches for bad blocks).
// Output k is S_k * eo_forward_scale(k), S_k = sum_n x_n cos((2n+1) k pi / 16); the scale factors are
// folded into the quantisation tables by the callers.
//
// Inverse (scipy's unnormalised DCT-III, out[n] = X_0 + 2 sum_k X_k cos(pi k (2n+1) / 16)): the mirror.
// Input k must be X_k * eo_inverse_prescale(k) (folded into the dequantisation table).
//
// T is float, double, the packed two-lane f2 (hic_f32x2.cuh) or the bound-carrying value of hic_dct_bound.h;
// eo_fma(a, b, c) = a * b + c in one rounding where the type has a fused operation.
// ------------------------------------------------------------------------------------------------
HIC_HD float eo_fma(float a, float b, float c) { return fmaf(a, b, c); }
HIC_HD double eo_fma(double a, double b, double c) { return fma(a, b, c); }

#define HIC_EO_T 0.41421356237309503445          /* tan(pi/8) */
/* ratios of c_m = cos(m pi/16): the odd rows of the forward matrix divided by their first entry */
#define HIC_EO_F13 0.84775906502257347697        /* c3/c1 */
#define HIC_EO_F15 0.56645449735052155749        /* c5/c1 */
#define HIC_EO_F17 0.19891236737965806158        /* c7/c1 */
#define HIC_EO_F37 0.23463313526982051971        /* c7/c3 */
#define HIC_EO_F31 1.17958042710327459801        /* c1/c3 */
#define HIC_EO_F35 0.66817863791929898998        /* c5/c3 */
#define HIC_EO_F51 1.76536686473017923049        /* c1/c5 */
#define HIC_EO_F57 0.35115330235708458462        /* c7/c5 */
#define HIC_EO_F53 1.49660576266548894786        /* c3/c5 */
#define HIC_EO_F75 2.84775906502257303288        /* c5/c7 */
#define HIC_EO_F73 4.26197262739566706813        /* c3/c7 */
#define HIC_EO_F71 5.02733949212584629862        /* c1/c7 */

// the part after the first butterflies: s_i = x_i + x_{7-i}, d_i = x_i - x_{7-i}
template <typename T>
HIC_HD void eo_forward8_tail(const T& s0, const T& s1, const T& s2, const T& s3, const T& d0, const T& d1, const T& d2,
                             const T& d3, T& x0, T& x1, T& x2, T& x3, T& x4, T& x5, T& x6, T& x7) {
    const T a = s0 + s3, p = s0 - s3, b = s1 + s2, q = s2 - s1;          // q = -(s1 - s2)
    x0 = a + b;
    x4 = a - b;                                                         // S_4 / cos(pi/4)
    x2 = eo_fma(T(-HIC_EO_T), q, p);                                    // S_2 / cos(pi/8)
    x6 = eo_fma(T(HIC_EO_T), p, q);                                     // S_6 / cos(pi/8)
    // odd part: S_k / cos(k pi/16)
    x1 = eo_fma(T(HIC_EO_F17), d3, eo_fma(T(HIC_EO_F15), d2, eo_fma(T(HIC_EO_F13), d1, d0)));
    x3 = eo_fma(T(-HIC_EO_F35), d3, eo_fma(T(-HIC_EO_F31), d2, eo_fma(T(-HIC_EO_F37), d1, d0)));
    x5 = eo_fma(T(HIC_EO_F53), d3, eo_fma(T(HIC_EO_F57), d2, eo_fma(T(-HIC_EO_F51), d1, d0)));
    x7 = eo_fma(T(-HIC_EO_F71), d3, eo_fma(T(HIC_EO_F73), d2, eo_fma(T(-HIC_EO_F75), d1, d0)));
}

template <typename T>
HIC_HD void eo_forward8(T& x0, T& x1, T& x2, T& x3, T& x4, T& x5, T& x6, T& x7) {
    const T s0 = x0 + x7, d0 = x0 - x7, s1 = x1 + x6, d1 = x1 - x6;
    const T s2 = x2 + x5, d2 = x2 - x5, s3 = x3 + x4, d3 = x3 - x4;
    eo_forward8_tail(s0, s1, s2, s3, d0, d1, d2, d3, x0, x1, x2, x3, x4, x5, x6, x7);
}

// in: X_k * eo_inverse_prescale(k).  Pivots (coefficient 1): X_1 in o0, X_5 in o1, X_3 in o2, X_7 in o3.
template <typename T>
HIC_HD void eo_inverse8(T& x0, T& x1, T& x2, T& x3, T& x4, T& x5, T& x6, T& x7) {
    const T A = x0 + x4, B = x0 - x4;
    const T C = eo_fma(T(HIC_EO_T), x6, x2);                            // in2 + t in6
    const T D = eo_fma(T(-HIC_EO_T), x2, x6);                           // in6 - t in2
    const T e0 = A + C, e3 = A - C, e1 = B - D, e2 = B + D;
    // odd part: every pivot entry is +-c1, so three ratios serve all twelve products
    const T o0 = eo_fma(T(-HIC_EO_F17), x7, eo_fma(T(-HIC_EO_F15), x5, eo_fma(T(-HIC_EO_F13), x3, x1)));
    const T o1 = eo_fma(T(HIC_EO_F15), x7, eo_fma(T(HIC_EO_F17), x3, eo_fma(T(HIC_EO_F13), x1, x5)));
    const T o2 = eo_fma(T(-HIC_EO_F13), x7, eo_fma(T(-HIC_EO_F17), x5, eo_fma(T(HIC_EO_F15), x1, x3)));
    const T o3 = eo_fma(T(-HIC_EO_F13), x5, eo_fma(T(HIC_EO_F15), x3, eo_fma(T(HIC_EO_F17), x1, x7)));
    x0 = e0 + o0;
    x7 = e0 - o0;
    x1 = e1 + o1;
    x6 = e1 - o1;
    x2 = e2 + o2;
    x5 = e2 - o2;
    x3 = e3 + o3;
    x4 = e3 - o3;
}

// Scale factors, derived by running the transforms above in double on unit vectors (so they cannot drift
// from the code): forward output k = S_k * eo_forward_scale(k); inverse input k = X_k * eo_inverse_prescale(k).
inline double eo_forward_scale(int k) {
    double x[8] = {1, 0, 0, 0, 0, 0, 0, 0};                     // S_k of the unit impulse at n = 0 is cos(k pi/16)
    eo_forward8(x[0], x[1], x[2], x[3], x[4], x[5], x[6], x[7]);
    return x[k] / cos(k * 3.14159265358979323846 / 16.0);
}
inline double eo_inverse_prescale(int k) {
    double x[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    x[k] = 1.0;
    eo_inverse8(x[0], x[1], x[2], x[3], x[4], x[5], x[6], x[7]);
    const double want = k == 0 ? 1.0 : 2.0 * cos(k * 3.14159265358979323846 / 16.0);      // coefficient of X_k in out[0]
    return want / x[0];
}

// ------------------------------------------------------------------------------------------------
// scaled decode: the m x m reduced inverse transform (m = 8 / s samples per block side, s = 2 or 4)
//
// B_s[k][0] = 1, B_s[k][n] = 2 D_s(n) cos(pi n (2k + 1) / (2m)), D_s(n) = sin(pi n s / 16) / (s sin(pi n / 16)):
// for a block whose coefficients are non-zero only at u, v < m, B_s X B_s^T is the mean of each s x s tile of
// the unrounded 8 x 8 IDCT.  Correctly rounded float64 values, row major [k][n]; tests/scaled_oracle.py holds
// the same bits and tests/test_scaled_host.py checks both against the closed form.
// ------------------------------------------------------------------------------------------------
#define HIC_SCALED_B4 { \
     0x1.0p+0,  0x1.cfefefc82ff2ap+0,  0x1.4e7ae9144f0fcp+0,  0x1.45d3819f43820p-1, \
     0x1.0p+0,  0x1.8056948c8d24bp-1, -0x1.4e7ae9144f0fcp+0, -0x1.894e984d2e2bcp+0, \
     0x1.0p+0, -0x1.8056948c8d24bp-1, -0x1.4e7ae9144f0fcp+0,  0x1.894e984d2e2bcp+0, \
     0x1.0p+0, -0x1.cfefefc82ff2ap+0,  0x1.4e7ae9144f0fcp+0, -0x1.45d3819f43820p-1 }
#define HIC_SCALED_B2 { \
     0x1.0p+0,  0x1.480d9d073b428p+0, \
     0x1.0p+0, -0x1.480d9d073b428p+0 }

// The definition of a scaled block, in float64: cq = the dequantised coefficients q[u][v] T[u][v], u, v < M, row
// major; rows first (A[u][k] = sum_v B[k][v] cq[u][v]), then columns (Y[j][k] = sum_u B[j][u] A[u][k]), every sum
// left to right from its first product, every product and sum rounded; out[j][k] = Y / 256 + 128, the value
// before the uint8 cast (wrap_u8).  The fix-up kernel and the CPU harness both run this.
template <int M>
HIC_HD void scaled_decoded_block(const int32_t* cq, double* out) {
    static_assert(M == 4 || M == 2, "scale 2 or 4");
    const double B4[16] = HIC_SCALED_B4, B2[4] = HIC_SCALED_B2;
    const double* B = M == 4 ? B4 : B2;
    double a[M * M];
#pragma unroll
    for (int u = 0; u < M; ++u)
#pragma unroll
        for (int k = 0; k < M; ++k) {
            double acc = dmul(B[M * k], (double)cq[M * u]);
#pragma unroll
            for (int v = 1; v < M; ++v) acc = dadd(acc, dmul(B[M * k + v], (double)cq[M * u + v]));
            a[M * u + k] = acc;
        }
#pragma unroll
    for (int j = 0; j < M; ++j)
#pragma unroll
        for (int k = 0; k < M; ++k) {
            double acc = dmul(B[M * j], a[k]);
#pragma unroll
            for (int u = 1; u < M; ++u) acc = dadd(acc, dmul(B[M * j + u], a[M * u + k]));
            out[M * j + k] = dadd(ddiv(acc, 256.0), 128.0);
        }
}

// The float32 fast path of the same transform, in place on v (M x M, row major): rows, then columns, each output a
// dense M-point sum acc = x_0 (B[k][0] = 1), then eo_fma(B[k][n], x_n, acc).  T is float, or the bound-carrying
// value of hic_dct_bound.h, which derives the error band of this code.
template <int M, typename T>
HIC_HD void scaled_transform(T* v) {
    static_assert(M == 4 || M == 2, "scale 2 or 4");
    const double B4[16] = HIC_SCALED_B4, B2[4] = HIC_SCALED_B2;
    const double* B = M == 4 ? B4 : B2;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        const int step = pass == 0 ? 1 : M, stride = pass == 0 ? M : 1;    // rows: v[M r + n]; columns: v[r + M n]
#pragma unroll
        for (int r = 0; r < M; ++r) {
            T x[M], y[M];
#pragma unroll
            for (int n = 0; n < M; ++n) x[n] = v[stride * r + step * n];
#pragma unroll
            for (int k = 0; k < M; ++k) {
                T acc = x[0];
#pragma unroll
                for (int n = 1; n < M; ++n) acc = eo_fma(T(B[M * k + n]), x[n], acc);
                y[k] = acc;
            }
#pragma unroll
            for (int k = 0; k < M; ++k) v[stride * r + step * k] = y[k];
        }
    }
}

// The near-tie bands.  A float32 quantised value C/q is trusted when its distance to the nearest
// half-integer exceeds kappa(u, v) * 4 u E / q (u = 2^-24, E = sum |x - 128| over the block); a float32
// decoded sample when its distance to the nearest integer (where the reference's uint8 truncation steps)
// exceeds 4 u / 256 * sum_k w_k |coef_k q_k| + 2^-15.  kappa(u, v) and w_k are RIGOROUS first-order bounds
// of the rounding error of the code above (hic_dct_bound.h), times HIC_BAND_MARGIN for everything of
// second order; blocks inside a band are redone in float64 by the fix-up kernels.
#define HIC_BAND_MARGIN 1.125

}  // namespace hic
