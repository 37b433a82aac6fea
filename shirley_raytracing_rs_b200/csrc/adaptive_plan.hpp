// adaptive_plan.hpp — tile-adaptive sampling (b200rt_render_adaptive): the pass schedule and the per-pixel error estimate.
// Pure arithmetic, compiled both into the merge kernel (render_kernel.cuh) and by g++ into tests/native/adaptive_plan_check.cpp,
// so the CPU test checks the exact arithmetic the device uses.
#pragma once
#include <cmath>
#include <cstdint>

#ifdef __CUDACC__
#define B200RT_HD __host__ __device__
#else
#define B200RT_HD
#endif

namespace b200rt {

// Samples every still-active tile has after pass k: n_k = min(initial * 2^k, max_samples).  Pass k renders [n_{k-1}, n_k)
// (n_{-1} = 0).  The first estimate is made after pass 1, so no selected pixel gets fewer than n_1 = min(2 * initial, max).
inline uint32_t adaptive_samples_after(uint32_t initial, uint32_t max_samples, uint32_t k) {
    uint64_t n = initial;
    for (uint32_t i = 0; i < k && n < max_samples; ++i) n *= 2;
    return n < max_samples ? (uint32_t)n : max_samples;
}

// Passes a tile that never meets the threshold runs: the first k with n_k == max_samples, plus pass 0.
inline uint32_t adaptive_max_passes(uint32_t initial, uint32_t max_samples) {
    uint32_t k = 0;
    while (adaptive_samples_after(initial, max_samples, k) < max_samples) ++k;
    return k + 1;
}

// e_p of one pixel from two independent means: F = the 2^-32 fixed-point sums of the n samples before the pass, P = those of the
// s samples of the pass.  Per channel, with every mean clamped at 1 like to_image (image.rs:34-40: a saturated channel has no error),
//   sigma = |F/n - P/s| * sqrt(n s) / (n + s)                the standard error of the combined mean
//   e     = sigma / (2 sqrt(max(m, 2^-16)))                  the same error after to_image's sqrt, in 0..1 output units
// and e_p is the largest channel's e.
B200RT_HD inline float adaptive_pixel_error(const long long* F, const long long* P, uint32_t n, uint32_t s) {
    const float inv = 1.0f / 4294967296.0f;
    const float fn = (float)n, fs = (float)s, ft = (float)n + (float)s;
    const float k = sqrtf(fn * fs) / ft;
    float e = 0.0f;
    for (int c = 0; c < 3; ++c) {
        const float a = fminf((float)F[c] * inv / fn, 1.0f);
        const float b = fminf((float)P[c] * inv / fs, 1.0f);
        const float m = fminf((float)(F[c] + P[c]) * inv / ft, 1.0f);
        const float sigma = fabsf(a - b) * k;
        e = fmaxf(e, sigma / (2.0f * sqrtf(fmaxf(m, 1.0f / 65536.0f))));
    }
    return e;
}

}  // namespace b200rt
