// Host-side check of tile-adaptive sampling's arithmetic (shirley_raytracing_rs_b200/csrc/adaptive_plan.hpp), compiled and run by
// tests/test_adaptive_plan.py.  It checks the pass schedule itself and prints the rest for the test to compare:
//   "sizeof <bytes>"   sizeof(B200rtAdaptiveParams)
//   then, for every line "n s F0 F1 F2 P0 P1 P2" on stdin, adaptive_pixel_error of those sums as "%.9g".
#include <algorithm>
#include <cstdio>
#include <vector>

#include "../../include/b200rt.h"
#include "../../shirley_raytracing_rs_b200/csrc/adaptive_plan.hpp"

using namespace b200rt;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { printf("  FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

static void expect_passes(uint32_t initial, uint32_t max_samples, const std::vector<uint32_t>& want) {
    const uint32_t passes = adaptive_max_passes(initial, max_samples);
    CHECK(passes == want.size());
    for (uint32_t k = 0; k < want.size(); ++k) CHECK(adaptive_samples_after(initial, max_samples, k) == want[k]);
    CHECK(adaptive_samples_after(initial, max_samples, passes + 3) == max_samples);      // capped for good
}

int main() {
    expect_passes(16, 2048, {16, 32, 64, 128, 256, 512, 1024, 2048});
    expect_passes(16, 100, {16, 32, 64, 100});
    expect_passes(16, 17, {16, 17});
    expect_passes(1, 2, {1, 2});
    expect_passes(3, 5, {3, 5});
    expect_passes(0x80000000u, 0xFFFFFFFFu, {0x80000000u, 0xFFFFFFFFu});   // no 32-bit wrap
    for (uint32_t initial = 1; initial < 70; ++initial)
        for (uint32_t max_samples = initial + 1; max_samples < 300; ++max_samples) {
            // the first estimate comes after pass 1: nobody stops below min(2 * initial, max)
            CHECK(adaptive_samples_after(initial, max_samples, 1) == std::min(2 * initial, max_samples));
            for (uint32_t k = 1; k < adaptive_max_passes(initial, max_samples); ++k)
                CHECK(adaptive_samples_after(initial, max_samples, k) > adaptive_samples_after(initial, max_samples, k - 1));
        }
    printf("schedule %s\n", failures ? "BAD" : "ok");
    printf("sizeof %zu\n", sizeof(B200rtAdaptiveParams));
    unsigned n, s;
    long long F[3], P[3];
    while (scanf("%u %u %lld %lld %lld %lld %lld %lld", &n, &s, &F[0], &F[1], &F[2], &P[0], &P[1], &P[2]) == 8)
        printf("%.9g\n", (double)adaptive_pixel_error(F, P, n, s));
    return failures ? 1 : 0;
}
