// hic_dct_bound.h -- rigorous float32 rounding-error bounds of the 8x8 transforms in hic_core.cuh, derived
// from THAT code: eo_forward8 / eo_inverse8 are templates, and here they run on a value type that carries,
// beside the exact linear form of every intermediate over the 64 inputs, a first-order bound of its
// accumulated rounding error.  Host only (library initialisation and the CPU test harness).
//
// Model.  A value n of the flow graph is n(x) = sum_i c_ni x_i.  A float32 operation returns the exact
// result times (1 + d), |d| <= u = 2^-24 (round to nearest; a fused multiply-add rounds once, so it is
// never worse than the separate pair bounded here), and a float32 constant is its exact value times
// (1 + d).  To first order the error of an output o is sum_n G_no d_n n(x), G_no the gain from node n to o, so
//
//   |err_o| <= u sum_n |G_no| |n(x)| <= u sum_i |x_i| sum_n |G_no| |c_ni|
//
// and, the sum of absolute values of linear forms being convex, <= u E max_i sum_n |G_no| |c_ni| with
// E = sum_i |x_i| (the maximum over the L1 ball sits on a vertex).  The per-input sums e_i travel forward
// through the graph, path gains in absolute value (no cancellation between rounding errors is assumed):
//
//   a +- b :  e = e(a) + e(b) + |c(a +- b)|
//   k * a  :  e = |k| e(a) + 2 |c(k a)|          (the product's rounding + the constant's own)
//
// Second-order terms are ~(depth * u) = 1e-6 of these; HIC_BAND_MARGIN (hic_core.cuh) covers them a
// hundred thousand times over.  tools/dct_error_bound.py derives the same numbers independently in Python
// (tests/test_oracle_dct.py compares), and the same test searches adversarially for blocks whose observed
// float32 error comes close to the bound.
#pragma once
#include <math.h>
#include "hic_core.cuh"

namespace hic {

struct BoundV {
    double c[64], e[64];
    bool is_const;
    double k;
    BoundV() : is_const(false), k(0.0) {
        for (int i = 0; i < 64; ++i) c[i] = e[i] = 0.0;
    }
    BoundV(double v) : is_const(true), k(v) {          // a constant of the algorithm: T(0.414...)
        for (int i = 0; i < 64; ++i) c[i] = e[i] = 0.0;
    }
};

inline BoundV bound_addsub(const BoundV& a, const BoundV& b, double sign) {
    BoundV r;
    for (int i = 0; i < 64; ++i) {
        r.c[i] = a.c[i] + sign * b.c[i];
        r.e[i] = a.e[i] + b.e[i] + fabs(r.c[i]);
    }
    return r;
}
inline BoundV operator+(const BoundV& a, const BoundV& b) { return bound_addsub(a, b, 1.0); }
inline BoundV operator-(const BoundV& a, const BoundV& b) { return bound_addsub(a, b, -1.0); }
inline BoundV eo_fma(const BoundV& k, const BoundV& x, const BoundV& y) {          // k * x + y, k a constant
    BoundV p;
    for (int i = 0; i < 64; ++i) {
        p.c[i] = k.k * x.c[i];
        p.e[i] = fabs(k.k) * x.e[i] + 2.0 * fabs(p.c[i]);
    }
    return p + y;
}

struct DctBounds {
    // forward: |C32 - C| <= kappa_fwd[8u+v] * 4 u E for coefficient (u, v) (C = the reference's unnormalised
    // DCT value, E = sum |x - 128|); includes the +1 of the rounded constant 4 / (scale_u scale_v q)
    double kappa_fwd[64];
    // inverse: |p32 - p| <= (4 u / 256) * sum_k w_inv[k] |coef_k q_k| for every sample p of the block
    // (k = 8u+v natural order; the maximum over the 64 samples is taken per input coefficient)
    double w_inv[64];
};

inline DctBounds dct_bounds() {
    DctBounds out;
    double sc[8], pre[8];
    for (int k = 0; k < 8; ++k) {
        sc[k] = eo_forward_scale(k);
        pre[k] = eo_inverse_prescale(k);
    }
    // ---- forward: rows, then columns (as K1) ----
    {
        static BoundV g[64];
        for (int i = 0; i < 64; ++i) {
            g[i] = BoundV();
            g[i].c[i] = 1.0;                               // x - 128: exact small integers, no input error
        }
        for (int r = 0; r < 8; ++r)
            eo_forward8(g[8 * r], g[8 * r + 1], g[8 * r + 2], g[8 * r + 3], g[8 * r + 4], g[8 * r + 5], g[8 * r + 6], g[8 * r + 7]);
        for (int c = 0; c < 8; ++c)
            eo_forward8(g[c], g[8 + c], g[16 + c], g[24 + c], g[32 + c], g[40 + c], g[48 + c], g[56 + c]);
        for (int u = 0; u < 8; ++u)
            for (int v = 0; v < 8; ++v) {
                double worst = 0.0;
                for (int i = 0; i < 64; ++i) worst = fmax(worst, g[8 * u + v].e[i]);
                // C = 4 S_uv = 4 b / (sc_u sc_v): the error of b in units of u E, turned into units of 4 u E of C
                out.kappa_fwd[8 * u + v] = worst / fabs(sc[u] * sc[v]) + 1.0;
            }
    }
    // ---- inverse: rows, then columns (as K7) ----
    {
        static BoundV g[64];
        for (int u = 0; u < 8; ++u)
            for (int v = 0; v < 8; ++v) {
                const int i = 8 * u + v;
                g[i] = BoundV();
                g[i].c[i] = pre[u] * pre[v] / 256.0;       // w = coef q * (pre_u pre_v / 256): float constant, rounded product
                g[i].e[i] = 2.0 * fabs(g[i].c[i]);
            }
        for (int r = 0; r < 8; ++r)
            eo_inverse8(g[8 * r], g[8 * r + 1], g[8 * r + 2], g[8 * r + 3], g[8 * r + 4], g[8 * r + 5], g[8 * r + 6], g[8 * r + 7]);
        for (int c = 0; c < 8; ++c)
            eo_inverse8(g[c], g[8 + c], g[16 + c], g[24 + c], g[32 + c], g[40 + c], g[48 + c], g[56 + c]);
        for (int k = 0; k < 64; ++k) {
            double worst = 0.0;
            for (int s = 0; s < 64; ++s) worst = fmax(worst, g[s].e[k]);
            out.w_inv[k] = worst * 256.0 / 4.0;
        }
    }
    return out;
}

// scaled decode (scaled_transform<M>): |p32 - p| <= (4 u / 256) sum_k w[k] |cq_k| + 2^-17 for every sample p = Y / 256
// + 128 of an M x M block, cq_k = q T of input k = M u + v (the maximum over the M x M samples per input).  The
// inputs cq / 256 are exact in float32 (|q T| < 2^22, a power-of-two scale); the final + 128 rounds once more, by at
// most u |Y / 256| + 2^-17, hence the |c| added to each output's sum.
template <int M>
inline void scaled_bounds(double* w) {
    static BoundV g[M * M];
    for (int i = 0; i < M * M; ++i) {
        g[i] = BoundV();
        g[i].c[i] = 1.0 / 256.0;
    }
    scaled_transform<M>(g);
    for (int k = 0; k < M * M; ++k) {
        double worst = 0.0;
        for (int s = 0; s < M * M; ++s) worst = fmax(worst, g[s].e[k] + fabs(g[s].c[k]));
        w[k] = worst * 256.0 / 4.0;
    }
}

}  // namespace hic
