// launch_plan.hpp — how a render or closest-hit launch is shaped: CTA size, shared-memory plan, sample-range schedule, grid.
// Pure host arithmetic (no CUDA calls), so tests/native/launch_plan_check.cpp runs it on the CPU.  Included by the device
// headers for the layout constants and SmemPlan, which the kernels' argument structs embed.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdint>

namespace b200rt {

constexpr int BLOCK = 256;          // threads per CTA of the parity-hook kernels (K1); the render kernel's CTA size is its BLK template argument (768 by default)
constexpr int TILE_W = 8, TILE_H = 4;   // one warp renders an 8x4 pixel tile, one lane per pixel
constexpr uint32_t MAX_CHUNKS = 64;     // sample ranges per tile
constexpr uint32_t RAYQ_SLOTS = 32, RAYQ_FIELDS = 9;   // v2: o, d, RNG state + stream, tile pixel
// Staged nodes are padded to SMEM_NODE_QUADS x 16 B (80 B instead of 64): with a 64-byte stride the quad k of every node falls
// into one of only two 16-byte bank groups (node parity), so the divergent LDS.128 of a quarter-warp collide; a stride of 5
// quads walks all eight groups (measured +1.2 % on the bench frame; padding the 32-byte geometry records to 48 B the same
// way measured 3 % slower).
constexpr int SMEM_NODE_QUADS = 5;

// The 8x4 tiles that cover rows [row_begin, row_end) of a W x H frame, (0, 0) meaning the whole frame.  `ok` is false for a
// range outside the image; an empty range covers no tile.
struct TileGrid { bool ok; uint32_t row_begin, row_end, tiles_x, tile_row0, n_tiles; };

inline TileGrid tile_grid(uint32_t W, uint32_t H, uint32_t row_begin, uint32_t row_end) {
    TileGrid g{};
    g.row_begin = row_begin;
    g.row_end = row_begin == 0 && row_end == 0 ? H : row_end;
    g.ok = g.row_end <= H && g.row_begin <= g.row_end;
    g.tiles_x = (W + TILE_W - 1) / TILE_W;
    g.tile_row0 = g.row_begin / TILE_H;
    g.n_tiles = g.ok && g.row_end > g.row_begin ? g.tiles_x * ((g.row_end + TILE_H - 1) / TILE_H - g.tile_row0) : 0u;
    return g;
}

struct SmemPlan {
    uint32_t all_in_smem;           // 1: nodes + geom + mats + tex all staged (SmemAcc)
    uint32_t n_top;                 // nodes staged when !all_in_smem
    uint32_t stack_depth;           // entries per thread
    uint32_t bytes;                 // dynamic shared memory per CTA
};

struct SceneSize { uint32_t n_nodes, n_prims, n_tex, bvh_depth; };

// shared-memory budget: stage the whole scene when it fits, else nothing (the L1 cache does better)
inline SmemPlan make_plan(const SceneSize& s, size_t smem_optin, uint32_t blocks_per_sm_target, uint32_t block_threads = BLOCK, size_t extra_bytes = 0) {
    SmemPlan p{};
    size_t budget = smem_optin / blocks_per_sm_target;
    if (budget > smem_optin) budget = smem_optin;
    budget = budget > 2048 ? budget - 1024 : budget;   // per-CTA reserved shared memory
    p.stack_depth = s.bvh_depth + 3;   // + the sentinel entry of the v2 kernel
    // per-thread stack columns + whatever else the kernel keeps per CTA
    size_t stack_bytes = (size_t)p.stack_depth * block_threads * sizeof(int) + extra_bytes;
    size_t scene_bytes = (size_t)s.n_nodes * (16 * SMEM_NODE_QUADS) + (size_t)s.n_prims * 64 + (size_t)s.n_tex * 32;
    if (scene_bytes + stack_bytes <= budget) {
        p.all_in_smem = 1; p.n_top = s.n_nodes;
        p.bytes = (uint32_t)(scene_bytes + stack_bytes);
    } else {
        // Scenes that do not fit: nothing is staged, every array is read through __ldg and the shared memory
        // left over is L1 cache (a staged prefix of the tree was measured slower — rt_device.cuh: GmemAcc).
        p.all_in_smem = 0;
        p.n_top = 0;
        p.bytes = (uint32_t)stack_bytes;
    }
    return p;
}

// The closest-hit kernel (and scene_info's bvh_nodes_in_smem): plan for two CTAs per SM, else one if that stages the scene.
inline SmemPlan hook_plan(const SceneSize& s, size_t smem_optin) {
    SmemPlan plan = make_plan(s, smem_optin, 2);
    if (!plan.all_in_smem) { SmemPlan p1 = make_plan(s, smem_optin, 1); if (p1.all_in_smem) plan = p1; }
    return plan;
}

// Whether a launch may test boxes with the centre-form slab test (rt_device.cuh: aabb_center2) instead of the exact
// Aabb::hit2 arithmetic.  `box_pad` is how far every BVH box was grown (scene_create: 4e-6 x max_abs_coord), `max_abs_coord`
// the largest |coordinate| of any primitive box, `max_origin` the largest |coordinate| of a ray origin and `min_dir_inf` the
// smallest max_k |d_k| over the rays (NaN or 0: never fast).  The centre form must be conservative, entering a box early but
// never culling a box the ray meets.  Let M = max(max_abs_coord, max_origin) and eps = 2^-23.
//  * Rounding.  A plane distance takes three roundings (-(o * inv), then the two FMAs) of values below |o|, |c| + |o| and
//    |c| + h + |o| in units of |inv|: at most eps / 2 x (3 |o| + 2 |c| + h) <= 3 eps M |inv| in all, against the pad of
//    >= 4 eps M |inv| the first condition asks for.  So a plane `pad` outside the primitive's box is computed at least
//    pad / 4 outside it.
//  * The reciprocal clamp.  On an axis whose |d_k| < 1e-18 the slab test takes |inv| = 1e18 (clamp_inv) instead of
//    1 / |d_k|, so its far plane comes in to (its distance in space) x 1e18.  A hit point p of the primitive has p_k inside
//    the primitive's box, so (say d_k > 0) the padded far plane is hi_k + pad - o_k >= pad + t d_k >= pad away from the
//    origin, and the computed far distance is at least pad / 4 x 1e18.  On the axis j of the largest |d_j|,
//    t |d_j| = |p_j - o_j| <= max_abs_coord + M.  So the clamp culls no hit while
//        |d|inf >= 4 (max_abs_coord + M) / (pad x 1e18),
//    about 1e-11 at the largest origin the first condition allows (M = 8.4 max_abs_coord), whatever the scene's scale.
//    Shorter directions (the reference's Ray is not normalised) take the exact path.
// tests/native/slab_guard_check.cpp runs the centre-form test on the CPU against the f64 box interval over this range.
inline bool fast_slab_ok(float box_pad, float max_abs_coord, float max_origin, float min_dir_inf) {
    const float M = std::max(max_abs_coord, max_origin);
    return box_pad >= 4.0f * 1.1920929e-7f * M
        && min_dir_inf > 0.0f && (double)min_dir_inf * box_pad * 1e18 >= 4.0 * ((double)max_abs_coord + M);
}

struct RenderShape { uint32_t block_threads; SmemPlan plan; };

// The path tracer runs one 768-thread CTA per SM (profiles/r02_experiments.md §16).  A deep tree (the device-built linear
// BVH can reach 40-50 levels) needs more stack per thread than 768 threads leave room for: fall back to smaller CTAs rather
// than fail.  (Only scenes that live in global memory get that deep; a scene that fits in shared memory runs 768 threads.)
inline RenderShape render_shape(const SceneSize& s, size_t smem_optin) {
    // per warp: the fixed-point tile sums and the primary-ray ring; per thread: 7 words of path state (attenuation, emitted, pixel)
    auto extra_for = [](uint32_t threads) { return (size_t)(threads / 32) * (96 * sizeof(long long) + RAYQ_FIELDS * RAYQ_SLOTS * sizeof(uint32_t)) + (size_t)threads * 7 * sizeof(float); };
    RenderShape r{768, make_plan(s, smem_optin, 1, 768, extra_for(768))};
    while (!r.plan.all_in_smem && r.plan.bytes + 1024 > smem_optin && r.block_threads > 256) {
        r.block_threads = r.block_threads > 512 ? 512 : 256;
        r.plan = make_plan(s, smem_optin, 1, r.block_threads, extra_for(r.block_threads));
    }
    return r;
}

struct SampleSchedule { uint32_t chunks; uint32_t chunk_begin[MAX_CHUNKS + 1]; };

// Work granularity (profiles/r02_experiments.md §2, §9, §17).  A tile's samples are split into sample ranges that SHRINK:
// the launch ends when the last item ends, so the last items must be small (a whole-tile item of the 1200x800 frame is
// ~1 ms: 5 % of a 63-spp launch, which is what one of 8 GPUs renders), while big items are cheaper per sample (a warp
// drains once per item).  Guided schedule: each range takes 70 % of what is left — at most `cap` samples, 7 % of a warp's
// share of the launch, so that frames with few tiles per warp (tile shards, small images) still balance — until the rest is
// below ~1.5x the target size of the last range, 0.2 % of a warp's share of the launch (2 % for scenes read through L1,
// where every extra item costs L1 locality and atomics: whole tiles on the config-4 frames).  Items are handed out
// range by range, bottom rows first within each.  Measured against uniform ranges: +2.9 % at 500 spp, +5.8 % at 63 spp,
// +4.7 % at 16 spp on the bench frame.  forced_chunks = n > 0 (B200RT_CHUNKS) splits the samples into n near-equal ranges
// instead, the first ones taking the remainder.
inline SampleSchedule sample_schedule(uint32_t samples, uint32_t my_tiles, uint32_t resident_warps, bool all_in_smem, int forced_chunks) {
    const uint32_t S = samples;
    const double tiles_per_warp = (double)my_tiles / (double)resident_warps;
    const double share = std::max((double)S * tiles_per_warp, 1e-9);                  // samples x tiles a resident warp renders
    const double last_target = std::max(1.0, (all_in_smem ? 0.002 : 0.02) * share);
    // no item above ~7 % of a warp's share (a heavy tile costs ~3x the average one) — but not below 8 samples (256 paths) either
    // when that share is small (tiny frames): an item drains the warp once whatever its size
    const double cap = std::max(std::max(1.0, 0.07 * share), std::min(8.0, 0.5 * share));
    uint32_t sizes[MAX_CHUNKS]; uint32_t C = 0;
    if (forced_chunks > 0) {
        C = (uint32_t)std::min<int64_t>(std::min<int64_t>(forced_chunks, MAX_CHUNKS), S);
        for (uint32_t k = 0; k < C; ++k) sizes[k] = S / C + (k < S % C ? 1u : 0u);
    } else {
        uint32_t rem = S;
        double cap_now = cap;
        while (rem > 0) {
            uint32_t s = (uint32_t)std::llround(std::min(cap_now, 0.7 * rem));
            s = std::min(std::max(s, 1u), rem);
            if (rem <= (uint32_t)std::ceil(1.5 * last_target) || C + 1 == MAX_CHUNKS) s = (C + 1 == MAX_CHUNKS || rem <= cap_now * 1.5) ? rem : s;
            sizes[C++] = s; rem -= s;
            if (C + 8 >= MAX_CHUNKS) cap_now = std::max(cap_now, (double)rem / 6.0);      // running out of table entries: bigger ranges
        }
    }
    if (C == 0) { sizes[0] = S; C = 1; }
    if ((uint64_t)my_tiles * C > 0xFFFFFFF0ull) { sizes[0] = S; C = 1; }      // the 32-bit work counter
    SampleSchedule r;
    r.chunks = C;
    r.chunk_begin[0] = 0;
    for (uint32_t k = 0; k < MAX_CHUNKS; ++k) r.chunk_begin[k + 1] = k < C ? r.chunk_begin[k] + sizes[k] : S;
    return r;
}

// CTAs to launch: the persistent grid, or fewer when there are fewer work items than resident warps.
inline uint32_t render_grid(uint32_t full_grid, uint32_t my_tiles, uint32_t chunks, uint32_t warps_per_block) {
    const uint64_t grid_needed = ((uint64_t)my_tiles * chunks + warps_per_block - 1) / warps_per_block;
    return grid_needed < full_grid ? std::max(1u, (uint32_t)grid_needed) : full_grid;
}

}  // namespace b200rt
