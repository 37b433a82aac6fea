// Host-side check of the launch policy (shirley_raytracing_rs_b200/csrc/launch_plan.hpp), compiled and run by
// tests/test_launch_plan.py.  An image is the same whatever the schedule, so the automatic sample-range schedules are
// pinned here to the values the guided schedule produced when it was measured (profiles/r02_experiments.md §17);
// a change to them shows up as a failure here rather than only as a slower bench line.
#include <cstdio>
#include <vector>

#include "../../shirley_raytracing_rs_b200/csrc/launch_plan.hpp"

using namespace b200rt;

static int failures = 0;
#define CHECK(cond) do { if (!(cond)) { printf("  FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); ++failures; } } while (0)

static void report(const char* what, int before) { printf("%s %s\n", what, failures == before ? "ok" : "BAD"); }

static void expect_schedule(const char* name, const SampleSchedule& s, const std::vector<uint32_t>& begin) {
    bool same = s.chunks + 1 == begin.size();
    for (size_t k = 0; same && k < begin.size(); ++k) same = s.chunk_begin[k] == begin[k];
    if (!same) {
        printf("  %s: got chunks %u begin {", name, s.chunks);
        for (uint32_t k = 0; k <= s.chunks; ++k) printf("%s%u", k ? ", " : "", s.chunk_begin[k]);
        printf("}\n");
    }
    CHECK(same);
}

// the properties every schedule has, automatic or forced
static void check_invariants(const SampleSchedule& s, uint32_t samples, uint32_t my_tiles) {
    CHECK(s.chunks >= 1 && s.chunks <= MAX_CHUNKS);
    CHECK((uint64_t)my_tiles * s.chunks <= 0xFFFFFFF0ull);
    CHECK(s.chunk_begin[0] == 0);
    for (uint32_t k = 0; k < s.chunks; ++k) CHECK(s.chunk_begin[k + 1] > s.chunk_begin[k]);   // no empty range
    for (uint32_t k = s.chunks; k <= MAX_CHUNKS; ++k) CHECK(s.chunk_begin[k] == samples);     // the ranges sum to samples
}

int main() {
    const uint32_t warps = 148 * 1 * 24;                       // B200: 148 SMs x one 768-thread CTA
    const uint32_t weekend = 150 * 200, c4 = 480 * 540, small = 12 * 16;   // 8x4 tiles of 1200x800, 3840x2160, 96x64
    {
        int before = failures;
        expect_schedule("weekend 500", sample_schedule(500, weekend, warps, true, 0), {0, 296, 439, 482, 495, 500});
        expect_schedule("weekend 63", sample_schedule(63, weekend, warps, true, 0), {0, 37, 55, 61, 63});
        expect_schedule("weekend 16", sample_schedule(16, weekend, warps, true, 0), {0, 9, 14, 16});
        expect_schedule("c4 64", sample_schedule(64, c4, warps, false, 0), {0, 64});
        expect_schedule("c4 64, 1/8 tile shard", sample_schedule(64, c4 / 8, warps, false, 0), {0, 41, 57, 64});
        expect_schedule("96x64 1", sample_schedule(1, small, warps, true, 0), {0, 1});
        std::vector<uint32_t> b64, b500;
        for (uint32_t k = 0; k <= 64; k += 2) b64.push_back(k);
        expect_schedule("96x64 64", sample_schedule(64, small, warps, true, 0), b64);
        for (uint32_t k = 0; k <= 448; k += 8) b500.push_back(k);
        for (uint32_t k : {457u, 466u, 475u, 484u, 493u, 498u, 500u}) b500.push_back(k);
        expect_schedule("96x64 500", sample_schedule(500, small, warps, true, 0), b500);
        report("automatic schedules", before);
    }
    {   // forced: n near-equal ranges, the first ones taking the remainder (as sharding.sample_ranges)
        int before = failures;
        expect_schedule("forced 1", sample_schedule(500, weekend, warps, true, 1), {0, 500});
        expect_schedule("forced 3", sample_schedule(500, weekend, warps, true, 3), {0, 167, 334, 500});
        expect_schedule("forced 5", sample_schedule(63, weekend, warps, true, 5), {0, 13, 26, 39, 51, 63});
        expect_schedule("forced 5 of 3 samples", sample_schedule(3, weekend, warps, true, 5), {0, 1, 2, 3});
        CHECK(sample_schedule(1000, weekend, warps, true, 100).chunks == MAX_CHUNKS);
        for (uint32_t S : {1u, 2u, 7u, 63u, 64u, 65u, 500u, 4096u})
            for (int n : {1, 2, 3, 5, 8, 63, 64, 100}) {
                SampleSchedule s = sample_schedule(S, weekend, warps, true, n);
                check_invariants(s, S, weekend);
                for (uint32_t k = 0; k < s.chunks; ++k) {
                    const uint32_t size = s.chunk_begin[k + 1] - s.chunk_begin[k];
                    CHECK(size == S / s.chunks + (k < S % s.chunks ? 1u : 0u));
                }
            }
        report("forced schedules", before);
    }
    {
        int before = failures;
        for (uint32_t S : {1u, 2u, 3u, 5u, 8u, 16u, 31u, 63u, 64u, 100u, 256u, 500u, 1000u, 4096u, 100000u, 0xFFFFFFFFu})
            for (uint32_t tiles : {1u, 7u, small, c4 / 8, weekend, c4, 1u << 26, 1u << 28})
                for (uint32_t w : {1u, 24u, 148u * 8, warps, 2 * warps})
                    for (bool smem : {false, true}) check_invariants(sample_schedule(S, tiles, w, smem, 0), S, tiles);
        CHECK(sample_schedule(4096, 1u << 28, warps, true, 0).chunks == 1);   // 2^28 tiles x 16 ranges would wrap the work counter
        report("schedule invariants", before);
    }
    {   // B200: 232 448 bytes of opt-in shared memory per CTA
        int before = failures;
        const size_t optin = 232448;
        RenderShape w = render_shape({485, 488, 490, 13}, optin);                // the Weekend final scene
        CHECK(w.block_threads == 768 && w.plan.all_in_smem == 1 && w.plan.n_top == 485 && w.plan.bytes + 1024 <= optin);
        RenderShape big = render_shape({999999, 1000000, 1000000, 30}, optin);   // 1e6 primitives, shallow tree
        CHECK(big.block_threads == 768 && big.plan.all_in_smem == 0 && big.plan.n_top == 0 && big.plan.stack_depth == 33);
        RenderShape d51 = render_shape({999999, 1000000, 1000000, 51}, optin);
        CHECK(d51.block_threads == 512 && d51.plan.all_in_smem == 0 && d51.plan.bytes + 1024 <= optin);
        CHECK(render_shape({999999, 1000000, 1000000, 50}, optin).block_threads == 768);
        RenderShape d90 = render_shape({999999, 1000000, 1000000, 90}, optin);
        CHECK(d90.block_threads == 256 && d90.plan.all_in_smem == 0 && d90.plan.bytes + 1024 <= optin);
        // the closest-hit kernel: two CTAs per SM when the scene fits twice, else one
        CHECK(hook_plan({485, 488, 490, 13}, optin).n_top == 485);
        CHECK(hook_plan({999999, 1000000, 1000000, 30}, optin).n_top == 0);
        report("render shape and hook plan", before);
    }
    {
        int before = failures;
        CHECK(render_grid(148, weekend, 5, 24) == 148);
        CHECK(render_grid(148, small, 1, 24) == 8);
        CHECK(render_grid(148, small, 32, 24) == 148);
        CHECK(render_grid(148, 0, 1, 24) == 1);
        report("render grid", before);
    }
    {
        int before = failures;
        TileGrid g = tile_grid(1200, 800, 0, 0);                      // (0, 0): the whole frame
        CHECK(g.ok && g.row_begin == 0 && g.row_end == 800 && g.tiles_x == 150 && g.tile_row0 == 0 && g.n_tiles == weekend);
        g = tile_grid(97, 61, 0, 0);                                  // ragged: partial tiles on the right and at the bottom
        CHECK(g.ok && g.row_end == 61 && g.tiles_x == 13 && g.n_tiles == 13 * 16);
        g = tile_grid(7, 3, 0, 3);
        CHECK(g.ok && g.tiles_x == 1 && g.n_tiles == 1);
        for (uint32_t r : {1u, 8u, 9u, 61u}) {                        // empty ranges cover no tile
            g = tile_grid(97, 61, r, r);
            CHECK(g.ok && g.n_tiles == 0 && g.row_begin == r && g.row_end == r);
        }
        g = tile_grid(97, 61, 5, 10);                                 // [5, 10) ends mid-tile: tile rows 1 and 2
        CHECK(g.ok && g.tile_row0 == 1 && g.n_tiles == 13 * 2);
        g = tile_grid(97, 61, 0, 62);                                 // outside the image
        CHECK(!g.ok && g.row_end == 62 && g.n_tiles == 0);
        g = tile_grid(97, 61, 10, 5);
        CHECK(!g.ok && g.n_tiles == 0);
        g = tile_grid(97, 61, 62, 0);
        CHECK(!g.ok && g.row_end == 0);
        // every non-empty range: the grid the render launch computed before it took it from tile_grid
        for (uint32_t W : {1u, 7u, 8u, 9u, 97u})
            for (uint32_t H : {1u, 3u, 4u, 5u, 61u})
                for (uint32_t r0 = 0; r0 < H; ++r0)
                    for (uint32_t r1 = r0 + 1; r1 <= H; ++r1) {
                        g = tile_grid(W, H, r0, r1);
                        const uint32_t tiles_x = (W + TILE_W - 1) / TILE_W, tile_row0 = r0 / TILE_H, tile_row1 = (r1 + TILE_H - 1) / TILE_H;
                        CHECK(g.ok && g.row_begin == r0 && g.row_end == r1 && g.tiles_x == tiles_x && g.tile_row0 == tile_row0 &&
                              g.n_tiles == tiles_x * (tile_row1 - tile_row0));
                    }
        report("tile grid", before);
    }
    return failures ? 1 : 0;
}
