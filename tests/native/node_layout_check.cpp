// Host-side check of the BVH node packing (shirley_raytracing_rs_b200/csrc/node_layout.hpp), compiled and run by
// tests/test_node_layout.py.  Over random, degenerate (lo == hi), empty (lo > hi, NaN) and non-finite child boxes:
//   "contain"  each child's [c - h, c + h], read back from the paired slots and rounded as the exact slab path rounds it,
//              contains [lo, hi]; an empty axis has h < 0 (never entered), an infinite one the always-entered box
//   "refs"     q3 carries both child references bit for bit, and its two spare slots are 0
//   "permuted" the node equals the previous (child-major) layout with its slots permuted, bit for bit
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <random>
#include <vector>

#include "../../shirley_raytracing_rs_b200/csrc/node_layout.hpp"

using namespace b200rt;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { printf("  FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

// The previous packing, child-major: child ch's c[k] at float 6 ch + k, its h[k] at 6 ch + 3 + k, the refs at 12 and 13.
static void old_pack(const float* q, float* o) {
    for (int ch = 0; ch < 2; ++ch) {
        const float* lo = q + 6 * ch; const float* hi = lo + 3;
        for (int k = 0; k < 3; ++k) {
            float c = 0.f, h = -1.f;
            if (lo[k] <= hi[k]) {
                c = 0.5f * lo[k] + 0.5f * hi[k];
                h = std::nextafterf(std::max(hi[k] - c, c - lo[k]), INFINITY);
                if (!std::isfinite(c) || !std::isfinite(h)) { c = 0.f; h = 3.0e38f; }
            }
            o[6 * ch + k] = c; o[6 * ch + 3 + k] = h;
        }
    }
    o[12] = q[12]; o[13] = q[13]; o[14] = q[14]; o[15] = q[15];
}

static uint32_t bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

int main() {
    std::mt19937 gen(20261020u);
    const float specials[] = {0.f, -0.f, 1.f, -1.f, 1e-3f, 3.5f, -7.25f, 1e6f, -1e6f, 1e30f, -1e30f, FLT_MAX, -FLT_MAX, FLT_MIN, -FLT_MIN,
                              1e-40f, -1e-40f, 3.0e38f, INFINITY, -INFINITY, NAN};
    const int NS = sizeof(specials) / sizeof(specials[0]);
    std::uniform_real_distribution<float> u(-1.f, 1.f);
    std::uniform_int_distribution<int> pick(0, 7), spec(0, NS - 1), expo(-20, 20);
    auto value = [&]() { return std::ldexp(u(gen), expo(gen)); };
    int n_empty = 0, n_unbounded = 0, n_degenerate = 0, n_plain = 0;
    const int before_contain = failures;
    int fail_refs = 0, fail_perm = 0;
    for (int it = 0; it < 400000; ++it) {
        float q[16];   // the builder's HostNode: lo0, hi0, lo1, hi1, bits(ref0), bits(ref1), 0, 0
        for (int b = 0; b < 2; ++b)
            for (int k = 0; k < 3; ++k) {
                float lo, hi;
                switch (pick(gen)) {
                    case 0: lo = hi = value(); break;                                        // degenerate
                    case 1: lo = value(); hi = value(); if (lo <= hi) std::swap(lo, hi); break;   // empty unless equal
                    case 2: lo = spec(gen) < NS / 2 ? specials[spec(gen)] : value(); hi = specials[spec(gen)]; break;
                    case 3: lo = specials[spec(gen)]; hi = specials[spec(gen)]; break;
                    default: lo = value(); hi = value(); if (lo > hi) std::swap(lo, hi); break;
                }
                q[6 * b + k] = lo; q[6 * b + 3 + k] = hi;
            }
        int ref0 = (int)gen(), ref1 = (int)gen();
        memcpy(&q[12], &ref0, 4); memcpy(&q[13], &ref1, 4);
        q[14] = q[15] = 0.f;
        float p[16];
        pack_node(q, q + 3, q + 6, q + 9, ref0, ref1, p);

        for (int ch = 0; ch < 2; ++ch)
            for (int k = 0; k < 3; ++k) {
                const float lo = q[6 * ch + k], hi = q[6 * ch + 3 + k];
                const float c = p[NODE_C + 2 * k + ch], h = p[NODE_H + 2 * k + ch];
                if (!(lo <= hi)) { CHECK(h < 0.f && c - h > c + h); ++n_empty; continue; }
                if (!std::isfinite(lo) || !std::isfinite(hi)) { CHECK(c == 0.f && h == 3.0e38f); ++n_unbounded; continue; }
                if (lo == hi) ++n_degenerate; else ++n_plain;
                CHECK(std::isfinite(c) && h >= 0.f);
                if (h == 3.0e38f && c == 0.f) { ++n_unbounded; continue; }   // c or h overflowed: always entered
                CHECK(c - h <= lo && c + h >= hi);
            }

        int fr = failures;
        CHECK(bits(p[NODE_REF]) == (uint32_t)ref0 && bits(p[NODE_REF + 1]) == (uint32_t)ref1 && bits(p[14]) == 0u && bits(p[15]) == 0u);
        fail_refs += failures - fr;

        float o[16];
        old_pack(q, o);
        int slot[16];
        for (int ch = 0; ch < 2; ++ch)
            for (int k = 0; k < 3; ++k) { slot[6 * ch + k] = NODE_C + 2 * k + ch; slot[6 * ch + 3 + k] = NODE_H + 2 * k + ch; }
        for (int i = 12; i < 16; ++i) slot[i] = i;
        bool same = true;
        for (int i = 0; i < 16; ++i) same = same && bits(o[i]) == bits(p[slot[i]]);
        int fp = failures;
        CHECK(same);
        fail_perm += failures - fp;
    }
    // every kind of axis was generated
    CHECK(n_empty > 1000 && n_unbounded > 1000 && n_degenerate > 1000 && n_plain > 1000);
    printf("contain %s\n", failures - fail_refs - fail_perm == before_contain ? "ok" : "BAD");
    printf("refs %s\n", fail_refs == 0 ? "ok" : "BAD");
    printf("permuted %s\n", fail_perm == 0 ? "ok" : "BAD");
    printf("axes empty %d unbounded %d degenerate %d plain %d\n", n_empty, n_unbounded, n_degenerate, n_plain);
    return failures ? 1 : 0;
}
