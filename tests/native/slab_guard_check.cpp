// Host-side check of the fast-slab guard (shirley_raytracing_rs_b200/csrc/launch_plan.hpp: fast_slab_ok), compiled and run
// by tests/test_slab_guard.py.  The centre-form slab test (rt_device.cuh: aabb_center2) is restated lane by lane with fmaf
// (each FFMA2 lane rounds like fmaf) on child boxes padded as scene_create pads them and packed by pack_node, with the ray
// constants of the traversal (__frcp_rn reciprocal clamped to +-1e18, nood = -(o * inv)).  Each ray is its own launch:
// max_origin = |o|inf, min_dir_inf = |d|inf.  Whenever the guard allows the fast form and the f64 interval of the UNPADDED
// box meets [t_min, t_max], the fast test must enter the box.
//   "pinned"  the short ray of two spheres at y = +-5: the fast form culls a box the ray meets, and the guard refuses it
//   "sweep"   box scales 1e-3 .. 1e6, origins up to the guard's origin limit, directions down to its direction limit,
//             components that are 0, subnormal or below the 1e-18 clamp, boxes thinner than the pad
//   "needed"  the same sweep below the direction limit does cull boxes: the direction term is not vacuous
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <random>

#include "../../shirley_raytracing_rs_b200/csrc/launch_plan.hpp"
#include "../../shirley_raytracing_rs_b200/csrc/node_layout.hpp"

using namespace b200rt;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { printf("  FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

struct Box { float lo[3], hi[3]; };
struct Ray { float o[3], d[3]; };

static float clamp_inv(float x) { return fminf(fmaxf(x, -1e18f), 1e18f); }

// aabb_center2 for child `ch` of the packed node q; returns whether the traversal enters it (setp.le lo, hi)
static bool fast_enters(const float q[16], int ch, const Ray& r, float t_min, float t_max) {
    float lo = t_min, hi = t_max;
    float nr[3], fr[3];
    for (int k = 0; k < 3; ++k) {
        const float inv = clamp_inv(1.0f / r.d[k]);
        const float nood = -(r.o[k] * inv);
        const float c = q[NODE_C + 2 * k + ch], h = q[NODE_H + 2 * k + ch];
        const float tc = fmaf(c, inv, nood);
        nr[k] = fmaf(-h, fabsf(inv), tc);
        fr[k] = fmaf(h, fabsf(inv), tc);
    }
    lo = fmaxf(fmaxf(nr[0], nr[1]), fmaxf(nr[2], t_min));
    hi = fminf(fminf(fr[0], fr[1]), fminf(fr[2], t_max));
    return lo <= hi;
}

// Does the ray meet the (unpadded) box within [t_min, t_max]?  f64 slabs with the exact reciprocal of the f32 direction.
static bool meets_f64(const Box& b, const Ray& r, double t_min, double t_max) {
    double lo = t_min, hi = t_max;
    for (int k = 0; k < 3; ++k) {
        const double o = r.o[k], d = r.d[k];
        if (d == 0.0) { if (o < b.lo[k] || o > b.hi[k]) return false; continue; }
        double t0 = (b.lo[k] - o) / d, t1 = (b.hi[k] - o) / d;
        if (t0 > t1) std::swap(t0, t1);
        lo = std::max(lo, t0); hi = std::min(hi, t1);
    }
    return lo <= hi;
}

static float max_abs_of(const Box* b, int n) {
    float m = 0.f;
    for (int i = 0; i < n; ++i) for (int k = 0; k < 3; ++k) m = std::max(m, std::max(fabsf(b[i].lo[k]), fabsf(b[i].hi[k])));
    return m;
}

// A two-child node as scene_create builds it: pad = 4e-6 x the scene's largest coordinate, both boxes grown by it.
struct Node { float q[16]; float pad, max_abs; };
static Node make_node(const Box& b0, const Box& b1, float max_abs) {
    Node n; n.max_abs = max_abs; n.pad = max_abs * 4e-6f;
    Box p[2] = {b0, b1};
    for (auto& b : p) for (int k = 0; k < 3; ++k) { b.lo[k] -= n.pad; b.hi[k] += n.pad; }
    pack_node(p[0].lo, p[0].hi, p[1].lo, p[1].hi, ~0, ~1, n.q);
    return n;
}

static float dir_inf(const Ray& r) { return std::max(fabsf(r.d[0]), std::max(fabsf(r.d[1]), fabsf(r.d[2]))); }
static float origin_inf(const Ray& r) { return std::max(fabsf(r.o[0]), std::max(fabsf(r.o[1]), fabsf(r.o[2]))); }

int main() {
    // ---- pinned: spheres (0, +-5, 0) of radius 1, o = (0.999, 0, 0), d = (0, 1e-15, 0) -----------------------------------
    {
        const Box s0 = {{-1, 4, -1}, {1, 6, 1}}, s1 = {{-1, -6, -1}, {1, -4, 1}};
        const Box both[2] = {s0, s1};
        const Node n = make_node(s0, s1, max_abs_of(both, 2));
        const Ray r = {{0.999f, 0.f, 0.f}, {0.f, 1e-15f, 0.f}};
        const bool meets = meets_f64(s0, r, 0.001, INFINITY);
        const bool enters = fast_enters(n.q, 0, r, 0.001f, INFINITY);
        const bool allowed = fast_slab_ok(n.pad, n.max_abs, origin_inf(r), dir_inf(r));
        CHECK(n.max_abs == 6.f && meets && !enters);      // the hole: the clamped far plane on x is ~1e15, the box at ~4e15
        CHECK(!allowed);
        // at 1e-10 the same ray is allowed, and the fast form enters
        const Ray r2 = {{0.999f, 0.f, 0.f}, {0.f, 1e-10f, 0.f}};
        CHECK(fast_slab_ok(n.pad, n.max_abs, origin_inf(r2), dir_inf(r2)) && fast_enters(n.q, 0, r2, 0.001f, INFINITY));
        printf("pinned %s\n", failures == 0 ? "ok" : "BAD");
    }

    // ---- sweep -------------------------------------------------------------------------------------------------------
    std::mt19937_64 gen(20261022u);
    std::uniform_real_distribution<double> u01(0.0, 1.0);
    auto uni = [&](double a, double b) { return a + (b - a) * u01(gen); };
    auto logu = [&](double a, double b) { return std::exp(uni(std::log(a), std::log(b))); };
    const float tiny[] = {0.f, -0.f, 1e-20f, -1e-20f, 1e-30f, -1e-30f, 1e-40f, -1e-45f};
    const int before = failures;
    long long checked = 0, clamped_axis = 0, near_limit = 0, culled_below = 0, below_met = 0;
    for (int it = 0; it < 300000; ++it) {
        const double S = std::pow(10.0, uni(-3.0, 6.0));               // scene scale
        Box b[2];
        for (auto& x : b)
            for (int k = 0; k < 3; ++k) {
                const double c = uni(-S, S);
                const int kind = (int)(u01(gen) * 4);
                // extents: ordinary, small, thinner than the pad (4e-6 S), zero
                const double e = kind == 0 ? uni(0.01, 0.5) * S : kind == 1 ? uni(1e-4, 1e-2) * S : kind == 2 ? uni(0.0, 2e-6) * S : 0.0;
                x.lo[k] = (float)(c - e); x.hi[k] = (float)(c + e);
            }
        const Node n = make_node(b[0], b[1], max_abs_of(b, 2));
        const int ch = (int)(u01(gen) * 2);
        const Box& box = b[ch];
        // the origin: within the guard's origin limit (pad >= 4 eps |o|: 8.39 x max_abs), sometimes inside the box's slab
        const double o_lim = n.pad / (4.0 * 1.1920929e-7) * 0.999;
        Ray r;
        double p[3];
        for (int k = 0; k < 3; ++k) p[k] = uni(box.lo[k], box.hi[k]);   // a target point in the box
        const double R = u01(gen) < 0.5 ? o_lim : uni(0.0, o_lim);
        for (int k = 0; k < 3; ++k) r.o[k] = (float)uni(-R, R);
        // the direction: towards the target, scaled so that |d|inf is at or above the guard's limit, or below it
        const bool below = u01(gen) < 0.25;
        double dv[3];
        for (int k = 0; k < 3; ++k) dv[k] = p[k] - (double)r.o[k];
        const int main_axis = (int)(u01(gen) * 3);
        for (int k = 0; k < 3; ++k)
            if (k != main_axis && u01(gen) < 0.5) { r.o[k] = (float)p[k]; dv[k] = 0.0; }        // in the slab: a tiny component below
        double m = std::max(std::fabs(dv[0]), std::max(std::fabs(dv[1]), std::fabs(dv[2])));
        if (m == 0.0) continue;
        const double M = std::max<double>(n.max_abs, origin_inf(r));
        const double limit = 4.0 * (n.max_abs + M) / ((double)n.pad * 1e18);
        const double target = below ? limit * logu(1e-6, 0.5) : limit * (u01(gen) < 0.3 ? 1.0 + 1e-6 : logu(1.0, 1e12));
        for (int k = 0; k < 3; ++k) r.d[k] = (float)(dv[k] / m * target);
        for (int k = 0; k < 3; ++k)
            if (k != main_axis && dv[k] == 0.0) r.d[k] = tiny[(int)(u01(gen) * 8)];
        const double t_min = u01(gen) < 0.5 ? 0.0 : 0.001, t_max = INFINITY;
        if (!meets_f64(box, r, t_min, t_max)) continue;
        const bool allowed = fast_slab_ok(n.pad, n.max_abs, origin_inf(r), dir_inf(r));
        const bool enters = fast_enters(n.q, ch, r, (float)t_min, (float)t_max);
        if (below) { ++below_met; if (!enters) ++culled_below; }
        if (!allowed) continue;
        ++checked;
        bool clamped = false;
        for (int k = 0; k < 3; ++k) clamped = clamped || fabsf(r.d[k]) < 1e-18f;
        clamped_axis += clamped;
        near_limit += dir_inf(r) < 2.0 * limit;
        if (!enters) {
            ++failures;
            if (failures - before <= 5)
                printf("  FAILED sweep: pad %g max_abs %g o (%g %g %g) d (%g %g %g) box [%g %g %g]-[%g %g %g] t_min %g\n", n.pad, n.max_abs,
                       r.o[0], r.o[1], r.o[2], r.d[0], r.d[1], r.d[2], box.lo[0], box.lo[1], box.lo[2], box.hi[0], box.hi[1], box.hi[2], t_min);
        }
    }
    CHECK(checked > 100000 && clamped_axis > 20000 && near_limit > 10000);
    printf("sweep %s\n", failures == before ? "ok" : "BAD");
    CHECK(culled_below > 100);
    printf("needed %s\n", culled_below > 100 ? "ok" : "BAD");
    printf("checked %lld clamped-axis %lld near-limit %lld; below the limit %lld of %lld met boxes culled\n", checked, clamped_axis,
           near_limit, culled_below, below_met);
    return failures ? 1 : 0;
}
