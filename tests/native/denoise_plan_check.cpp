// Host-side check of the denoiser's arithmetic (shirley_raytracing_rs_b200/csrc/denoise_plan.hpp), compiled and run by
// tests/test_denoise_plan.py.  It prints, for the test to compare:
//   "sizeof <bytes>"   sizeof(B200rtDenoiseParams)
//   "taps <sum of the B3 weights> <sum of the 3x3 Gaussian>"
//   then, for every line of 22 numbers on stdin
//     lp lq vbar  np.xyz zp  nq.xyz zq  ap.rgb  aq.rgb  dist  la lb na nb
//   "<edge weight> <two-halves variance>" as "%.9g %.9g".
#include <cmath>
#include <cstdio>

#include "../../include/b200rt.h"
#include "../../shirley_raytracing_rs_b200/csrc/denoise_plan.hpp"

using namespace b200rt;

int main() {
    printf("sizeof %zu\n", sizeof(B200rtDenoiseParams));
    double b3 = 0.0, g3 = 0.0;
    for (int dy = -2; dy <= 2; ++dy) for (int dx = -2; dx <= 2; ++dx) b3 += (double)dn_b3(dx) * dn_b3(dy);
    for (int dy = -1; dy <= 1; ++dy) for (int dx = -1; dx <= 1; ++dx) g3 += (double)dn_g3(dx) * dn_g3(dy);
    printf("taps %.9g %.9g\n", b3, g3);
    float v[22];
    for (;;) {
        for (int i = 0; i < 22; ++i) if (scanf("%f", &v[i]) != 1) return 0;
        const float lscale = DN_SIGMA_L * sqrtf(fmaxf(v[2], 0.0f)) + DN_EPS_L;
        const float w = dn_edge_weight(v[0], v[1], lscale, v[3], v[4], v[5], v[6], v[7], v[8], v[9], v[10],
                                       v[11], v[12], v[13], v[14], v[15], v[16], v[17]);
        printf("%.9g %.9g\n", (double)w, (double)dn_two_halves_variance(v[18], v[19], v[20], v[21]));
    }
}
