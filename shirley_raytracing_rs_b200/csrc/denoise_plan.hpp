// denoise_plan.hpp — the arithmetic of the feature-guided à-trous denoiser (b200rt_render_denoised, b200rt_denoise).
// Pure arithmetic, compiled both into the filter kernels (denoise_kernels.cuh) and by g++ into tests/native/denoise_plan_check.cpp,
// so the CPU test checks the exact arithmetic the device uses.
//
// Method: the edge-avoiding à-trous wavelet filter (Dammertz et al. 2010) with the variance-guided luminance edge-stop of SVGF
// (Schied et al. 2017), on two independent half renders A and B of the same pixels ({sum rgb, count} float4 each) and the
// per-pixel features of a primary-hit pass: the mean face-flipped normal N, the mean hit distance z (0: every feature ray
// missed) and the mean first-hit albedo alb.  Per pixel p, with n = n_A + n_B:
//   c_p   = (A.rgb + B.rgb) / n                                             mean radiance
//   x_p   = c_p / max(alb_p, EPS_ALBEDO)                                   demodulated, per channel
//   v_p   = (l(A.rgb / n_A / alb') - l(B.rgb / n_B / alb'))^2 n_A n_B / n^2  two-halves variance of the luminance l of x_p
//                                                                             (alb' = max(alb_p, EPS_ALBEDO); 0 if n_A or n_B is 0)
// Iteration i = 0 .. iterations-1 (step s = 2^i) over the 5x5 taps q = p + s (dx, dy), dx, dy in -2..2, inside the frame:
//   vbar_p = the 3x3 Gaussian (1/4, 1/2, 1/4)^2 of v around p, at step 1, edge pixels repeated
//   w_pq   = h(dx) h(dy) * wl * wn * wz * wa,    h = (1/16, 1/4, 3/8, 1/4, 1/16)                        (B3 spline)
//   wl     = exp(-|l(x_p) - l(x_q)| / (SIGMA_L sqrt(vbar_p) + EPS_L))                                   luminance
//   wn     = max(0, N_p.N_q / (|N_p| |N_q|))^SIGMA_N   (0 when either normal is 0)                       normal
//   wz     = exp(-|z_p - z_q| / (SIGMA_Z max(z_p, z_q) s max(|dx|, |dy|)))                              relative depth
//   wa     = exp(-(|alb_p - alb_q|_1) / SIGMA_A)                                                        albedo
//   w_pq   = 0 when exactly one of p, q has z = 0; the centre tap's weight is h(0)^2 = 9/64 by definition.
//   x'_p   = sum_q w_pq x_q / sum_q w_pq           v'_p = sum_q w_pq^2 v_q / (sum_q w_pq)^2
// Remodulation: out_p = {x_p max(alb_p, EPS_ALBEDO) n, n}, the accumulation layout {mean * n, n}.  A pixel whose feature rays all
// missed (z = 0, the sky) keeps its own sums: out_p = {A.rgb + B.rgb, n}.
// Invariants the tests rely on:
//   * the centre tap always has weight 9/64 > 0, so sum_q w_pq > 0;
//   * the taps are summed in a fixed order (dy, then dx, ascending), so the output is deterministic;
//   * with zero variance a region of constant colour is returned unchanged to float rounding (wl = exp(0) = 1 between equal
//     luminances, and every x_q in the sum is the same value);
//   * a pixel whose feature rays all missed neither gives weight to nor takes weight from a pixel that hit something.
#pragma once
#include <cmath>
#include <cstdint>

#ifdef __CUDACC__
#define B200RT_DN_HD __host__ __device__
#else
#define B200RT_DN_HD
#endif

namespace b200rt {

constexpr float DN_EPS_ALBEDO = 1e-3f;   // albedo floor of the demodulation (black surfaces keep their radiance)
constexpr float DN_SIGMA_L = 4.0f;       // luminance edge-stop, in standard deviations (SVGF's sigma_l)
constexpr float DN_EPS_L = 1e-10f;       // keeps the luminance stop defined at zero variance
constexpr float DN_SIGMA_N = 128.0f;     // normal edge-stop exponent (SVGF's sigma_n)
constexpr float DN_SIGMA_Z = 0.05f;      // relative depth change allowed per pixel of tap distance
constexpr float DN_SIGMA_A = 0.1f;       // albedo edge-stop, L1 distance of the albedos
constexpr int DN_MAX_ITERATIONS = 5;

B200RT_DN_HD inline float dn_b3(int d) { return d == 0 ? 0.375f : (d == 1 || d == -1 ? 0.25f : 0.0625f); }
B200RT_DN_HD inline float dn_g3(int d) { return d == 0 ? 0.5f : 0.25f; }
B200RT_DN_HD inline float dn_luminance(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }
B200RT_DN_HD inline float dn_albedo_floor(float a) { return fmaxf(a, DN_EPS_ALBEDO); }

// v_p from the two halves' demodulated luminances la = l(A.rgb / n_a / alb'), lb = l(B.rgb / n_b / alb'): the square of
// adaptive_pixel_error's two-means estimate sigma = |a - b| sqrt(n_a n_b) / (n_a + n_b), taken before the gamma step.
B200RT_DN_HD inline float dn_two_halves_variance(float la, float lb, float na, float nb) {
    if (!(na > 0.0f) || !(nb > 0.0f)) return 0.0f;
    const float d = la - lb, t = na + nb;
    return d * d * (na * nb) / (t * t);
}

// The edge-stopping weight of a non-centre tap q of p, without the B3 factor.  np4 / nq4 = (N.xyz, z), ap / aq = albedo,
// dist = s max(|dx|, |dy|) >= 1, lscale = SIGMA_L sqrt(vbar_p) + EPS_L.
B200RT_DN_HD inline float dn_edge_weight(float lp, float lq, float lscale,
                                         float npx, float npy, float npz, float zp, float nqx, float nqy, float nqz, float zq,
                                         float apr, float apg, float apb, float aqr, float aqg, float aqb, float dist) {
    if ((zp == 0.0f) != (zq == 0.0f)) return 0.0f;   // sky against geometry: never mixed
    const float wl = expf(-fabsf(lp - lq) / lscale);
    const float nn = (npx * npx + npy * npy + npz * npz) * (nqx * nqx + nqy * nqy + nqz * nqz);
    const float c = nn > 0.0f ? fminf((npx * nqx + npy * nqy + npz * nqz) / sqrtf(nn), 1.0f) : 0.0f;
    const float wn = c > 0.0f ? powf(c, DN_SIGMA_N) : 0.0f;
    const float zm = fmaxf(zp, zq);
    const float wz = zm > 0.0f ? expf(-fabsf(zp - zq) / (DN_SIGMA_Z * zm * dist)) : 1.0f;
    const float wa = expf(-(fabsf(apr - aqr) + fabsf(apg - aqg) + fabsf(apb - aqb)) / DN_SIGMA_A);
    return wl * wn * wz * wa;
}

}  // namespace b200rt
