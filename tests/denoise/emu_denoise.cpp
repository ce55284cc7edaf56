// emu_denoise.cpp -- TEST HELPER: host (g++) build of the denoiser's per-pixel functions (csrc/sqt_denoise.cuh), run in
// the order the kernels run them (k_denoise_prep, then one k_denoise_level per level), so that tests can compare the
// device's bits with it and the formula of include/sqt.h with a numpy evaluation.
#include <vector>

#include "../../squigly-trace_b200/csrc/sqt_denoise.cuh"

using namespace sqt;

extern "C" {

// cv[p] = (c, v) of pixel p after k samples; counts may be NULL (every pixel has k samples), 0 entries mean k
void emu_denoise_input(long long npix, const float *s1, const float *s2, int k, const int *counts, float4 *cv) {
    for (long long i = 0; i < npix; ++i) {
        const int c = counts ? counts[i] : 0;
        cv[i] = denoise_input(s1 + 3 * i, s2 + 3 * i, c ? c : k);
    }
}

// one level of step s on cv (rows x cols) into out
void emu_denoise_level(int rows, int cols, const float4 *cv, const float4 *feat, const int2 *sk, int s, float sigma_l, float sigma_z,
                       float4 *out) {
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) out[(size_t)y * cols + x] = denoise_level_pixel(cv, feat, sk, rows, cols, y, x, s, sigma_l, sigma_z);
}

// `levels` levels of the filter on cv (rows x cols); the last level's (c, v) goes to out
void emu_denoise_levels(int rows, int cols, const float4 *cv, const float4 *feat, const int2 *sk, int levels, float sigma_l,
                        float sigma_z, float4 *out) {
    const long long npix = (long long)rows * cols;
    std::vector<float4> a(cv, cv + npix), b((size_t)npix);
    for (int i = 0; i < levels; ++i) {
        emu_denoise_level(rows, cols, a.data(), feat, sk, 1 << i, sigma_l, sigma_z, b.data());
        a.swap(b);
    }
    for (long long i = 0; i < npix; ++i) out[i] = a[i];
}

}
