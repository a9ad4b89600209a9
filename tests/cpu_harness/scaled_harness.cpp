// CPU check harness of the scaled decode: runs K7S's float32 arithmetic and the float64 definition the fix-up
// kernel runs (scaled_transform / scaled_decoded_block in hic_core.cuh, scaled_bounds in hic_dct_bound.h) on the
// host, so tests/test_scaled_host.py can compare them with tests/scaled_oracle.py without a GPU.  TEST
// INFRASTRUCTURE ONLY -- it is not linked into libhiccup_b200.so and nothing under hiccup_b200/ loads it.
// Build: g++ -O2 -ffp-contract=off -std=c++17 -shared -fPIC scaled_harness.cpp -o libhic_scaled_harness.so
#include "../../hiccup_b200/csrc/hic_core.cuh"
#include "../../hiccup_b200/csrc/hic_dct_bound.h"

using namespace hic;

static const int LUM[64] = HIC_LUM_TABLE;
static const int CHROMA[64] = HIC_CHROMA_TABLE;
static const uint8_t ZZ[64] = HIC_ZIGZAG8;

template <int M>
static void scaled_blocks(const int16_t* coef, int nb, int kind, uint8_t* out, uint8_t* flagged, double* ratio, uint8_t* exact) {
    const int* q = kind == 0 ? LUM : CHROMA;
    constexpr int ENTRIES = M == 4 ? 32 : 8;         // the scan entries K7S loads
    double w[M * M];
    scaled_bounds<M>(w);
    float sqw[M * M];
    for (int u = 0; u < M; ++u)
        for (int v = 0; v < M; ++v) sqw[M * u + v] = (float)(q[8 * u + v] * w[M * u + v] * HIC_BAND_MARGIN);
    const float MAGIC = 12582912.0f;
    for (int b = 0; b < nb; ++b) {
        const int16_t* c = coef + 64 * b;
        float v[M * M];
        int32_t cq[M * M];
        float energy = 0.f;
        double S_exact = 0.0;
        int ac = 0;
        for (int k = 0; k < ENTRIES; ++k) {
            const int nat = ZZ[k], u = nat >> 3, x = nat & 7;
            if (u >= M || x >= M) continue;
            v[M * u + x] = (float)(c[k] * q[nat]) * (1.f / 256.f);
            cq[M * u + x] = c[k] * q[nat];
            energy = fmaf(fabsf((float)c[k]), sqw[M * u + x], energy);
            S_exact += fabs((double)c[k]) * q[nat] * w[M * u + x];
            if (k) ac |= c[k];
        }
        double p64[M * M];
        scaled_decoded_block<M>(cq, p64);
        scaled_transform<M>(v);
        float margin = 1e30f;
        double worst = 0.0;
        for (int i = 0; i < M * M; ++i) {
            const float p = v[i] + 128.f;
            const float r = (p + MAGIC) - MAGIC;
            margin = fminf(margin, fabsf(p - r));
            out[M * M * b + i] = (uint8_t)((int)p & 0xFF);
            exact[M * M * b + i] = wrap_u8(p64[i]);
            if (S_exact > 0.0) {
                // the bound: (4 u / 256) sum w |cq| + 2^-17 (the constant 128's share of the final rounding)
                const double r64 = (fabs((double)p - p64[i]) - 7.62939453125e-6) / (4.0 / 16777216.0 / 256.0 * S_exact);
                if (r64 > worst) worst = r64;
            }
        }
        const float band = (float)(4.0 / 16777216.0 / 256.0) * energy + 3.0517578125e-5f;
        flagged[b] = ac != 0 && margin <= band;
        ratio[b] = worst;
    }
}

extern "C" {

// The committed basis B_s (m = 4: scale 2, m = 2: scale 4; row major m x m).
void hx_scaled_basis(int m, double* out) {
    const double b4[16] = HIC_SCALED_B4, b2[4] = HIC_SCALED_B2;
    for (int i = 0; i < m * m; ++i) out[i] = m == 4 ? b4[i] : b2[i];
}

// K7S's float32 path on the host.  coef: [nb][64] int16 scan order; out: [nb][m m] uint8 before the fix-up; flagged:
// [nb] 1 where K7S records the block; ratio: [nb] max over samples of the observed float32 error as a fraction of the
// rigorous bound (must stay below 1); exact: [nb][m m] the float64 definition (scaled_decoded_block).
void hx_scaled_blocks(const int16_t* coef, int nb, int kind, int m, uint8_t* out, uint8_t* flagged, double* ratio, uint8_t* exact) {
    if (m == 4) scaled_blocks<4>(coef, nb, kind, out, flagged, ratio, exact);
    else scaled_blocks<2>(coef, nb, kind, out, flagged, ratio, exact);
}

}  // extern "C"
