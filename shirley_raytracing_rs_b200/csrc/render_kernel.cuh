// render_kernel.cuh — K2: kernel arguments, scene staging and the persistent path-tracing kernel (path_trace_kernel_v2), the default
// (included by b200rt.cu; everything lives in namespace b200rt)
#pragma once
#include "adaptive_plan.hpp"
#include "rt_device.cuh"

namespace b200rt {

// ------------------------------------------------------------------------------------------
// kernel arguments
// ------------------------------------------------------------------------------------------
constexpr size_t LBVH_AUTO_MIN = 262144;   // primitives from which scene_create builds the tree on the device

struct Counters {                   // device-side, one per in-flight render
    unsigned long long rays, paths, nodes, prims, exhausted;
    unsigned int tile_counter, pad;
    unsigned long long diag[8];
};

struct RenderArgs {
    DeviceScene scene;
    DeviceCamera cam;
    SmemPlan plan;
    RngKeys keys;
    uint32_t samples, sample_offset, max_depth;
    uint32_t row_begin, row_end;
    uint32_t tiles_x, tile_row0, n_tiles;       // tile grid covering [row_begin, row_end)
    uint32_t shard_count, shard_index;
    uint32_t accumulate;
    uint32_t chunks;                            // work item = (tile, one of `chunks` contiguous sample ranges)
    // Items are handed out chunk by chunk (all tiles' first ranges, then all second ones, ...) and the ranges SHRINK
    // (chunk_begin[k] .. chunk_begin[k + 1]): big items while the grid is full, small ones at the end of the launch, where the
    // last items to finish decide how long the other SMs idle.  my_tiles = this shard's tiles.
    uint32_t my_tiles;
    uint32_t chunk_begin[MAX_CHUNKS + 1];
    long long* fix;                             // non-NULL: the sums are added to these per-pixel 2^-32 fixed-point sums [H][W][3] in global memory
                                                // (plain renders: when chunks > 1, finalize_kernel converts; adaptive passes: the pass buffer)
    const uint32_t* tile_list;                  // non-NULL: item j renders tile tile_list[j % my_tiles] (adaptive passes: the active tiles)
    uint32_t lim_samples;                       // acc_add's clamp is 2e9 / lim_samples: `samples` for plain renders, max_samples for adaptive passes
    uint32_t trav_threshold;                    // leave the traversal loop when fewer lanes than this still traverse
    uint32_t regen_min;                         // hand out new paths only when at least this many lanes are free
    float4* accum;
    Counters* counters;
};

// Stage the scene (or the top of the BVH) into shared memory and set up the accessor.
// Shared layout: [nodes][geom][mats][tex][stack: stack_depth x BLOCK ints]
template <class Acc> struct Stager;
template <> struct Stager<SmemAcc> {
    static __device__ __forceinline__ SmemAcc stage(const DeviceScene& s, const SmemPlan& plan, float4* smem, int** stack) {
        uint32_t n_nodes4 = s.n_nodes * 4, n_geom4 = s.n_prims * 2, n_mat4 = s.n_prims * 2, n_tex4 = s.n_tex * 2;
        float4* nodes = smem;
        float4* geom = nodes + s.n_nodes * SMEM_NODE_QUADS;
        float4* mats = geom + n_geom4;
        float4* tex = mats + n_mat4;
        const float4* gn = reinterpret_cast<const float4*>(s.nodes);
        const float4* gg = reinterpret_cast<const float4*>(s.geom);
        const float4* gm = reinterpret_cast<const float4*>(s.mats);
        const float4* gt = reinterpret_cast<const float4*>(s.tex);
        for (uint32_t i = threadIdx.x; i < n_nodes4; i += blockDim.x) nodes[(i >> 2) * SMEM_NODE_QUADS + (i & 3u)] = __ldg(gn + i);
        for (uint32_t i = threadIdx.x; i < n_geom4; i += blockDim.x) geom[i] = __ldg(gg + i);
        for (uint32_t i = threadIdx.x; i < n_mat4; i += blockDim.x) mats[i] = __ldg(gm + i);
        for (uint32_t i = threadIdx.x; i < n_tex4; i += blockDim.x) tex[i] = __ldg(gt + i);
        *stack = reinterpret_cast<int*>(tex + n_tex4);
        __syncthreads();
        SmemAcc a; a.nodes = nodes; a.geom = geom; a.mats = mats; a.tex = tex;
        return a;
    }
};
template <> struct Stager<GmemAcc> {
    static __device__ __forceinline__ GmemAcc stage(const DeviceScene& s, const SmemPlan& plan, float4* smem, int** stack) {
        *stack = reinterpret_cast<int*>(smem);     // nothing staged: shared memory holds only the per-CTA working arrays
        GmemAcc a;
        a.nodes = reinterpret_cast<const float4*>(s.nodes); a.geom = reinterpret_cast<const float4*>(s.geom);
        a.mats = reinterpret_cast<const float4*>(s.mats); a.tex = reinterpret_cast<const float4*>(s.tex);
        return a;
    }
};

// Per-pixel sums as 64-bit fixed point (2^-32) in shared memory: integer adds commute, so the
// result does not depend on which lane traced which sample, nor on scheduling or sharding.
// Contract (INTEGRATION.md): a sample whose radiance is NaN or infinite contributes nothing (the reference would
// carry the NaN into the pixel, which to_image writes as 0).  Each channel of a finite sample is clamped to +-`lim` =
// 2e9 / samples-per-call (adaptive passes: 2e9 / max_samples, over all passes), so a pixel's 2^-32 fixed-point sum (63 bits: |sum| < 2^31 = 2.1e9) cannot wrap whatever the
// emitters' strength; a clamped sample still saturates the pixel (to_image clips the mean at 1).
// The 64-bit add is two native 32-bit shared-memory atomics (low word with the old value returned, then the high word
// plus the carry, skipped when both are zero — the usual case: samples below 1.0 have no high word): integer adds
// commute and every carry is counted exactly once, so the sum is the same 64-bit integer whatever the order.
// (atomicAdd on a 64-bit shared word compiles to a compare-and-swap loop, ATOMS.CAST.SPIN.64: 3.5 % of the kernel's
// issue slots at 6-10 lanes.)
__device__ __forceinline__ void acc_add64(uint32_t word_addr, long long x) {
    const uint32_t lo = (uint32_t)x, hi = (uint32_t)((unsigned long long)x >> 32);
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(word_addr), "r"(lo) : "memory");
    const uint32_t up = hi + ((old + lo) < lo ? 1u : 0u);
    if (up) asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(word_addr + 4u), "r"(up) : "memory");
}
__device__ __forceinline__ void acc_add(long long* acc, uint32_t pixel, float3 v, float lim) {
    const float S = 4294967296.0f;
    // one test: any NaN or infinity makes the sum NaN or infinite (radiance is non-negative; the quarter keeps a finite triple finite)
    if (fabsf(fmaf(v.x, 0.25f, fmaf(v.y, 0.25f, v.z * 0.25f))) <= 3.0e38f) {
        v.x = fminf(fmaxf(v.x, -lim), lim); v.y = fminf(fmaxf(v.y, -lim), lim); v.z = fminf(fmaxf(v.z, -lim), lim);
        const uint32_t a0 = (uint32_t)__cvta_generic_to_shared(acc + pixel * 3);
        acc_add64(a0, __float2ll_rn(v.x * S));
        acc_add64(a0 + 8u, __float2ll_rn(v.y * S));
        acc_add64(a0 + 16u, __float2ll_rn(v.z * S));
    }
}

// ------------------------------------------------------------------------------------------
// K2: the persistent path-tracing kernel (render_scanline + ray_color, render.rs:17-70).
// Grid = one CTA of BLK threads per SM; every warp pulls work items — an 8x4-pixel tile and one of `chunks` ranges of
// its samples — from a global counter (bottom rows first: the geometry-heavy tiles are scheduled before the cheap sky
// tiles) and works through the item's (pixel, sample) list with all 32 lanes.  ncu on the first, straight-loop design
// (round 1, git history) showed 8.1 of 32 lanes active per instruction — inner-node visits at 13 lanes, leaf tests at 4,
// the marble texture at 2.7 — so this kernel is organised around lane utilisation, instruction count and registers:
//  * one outer iteration = shade the lanes whose traversal finished -> hand new paths to the free lanes once at least
//    `regen_min` of them are (from a per-warp ring of primary rays generated 32 at a time) -> ONE shared per-segment
//    set-up for both groups (IEEE reciprocals, scene-spanning primitives tested up front) -> traverse;
//  * state that is touched once per bounce (ray_color's attenuation and emitted accumulators, the path's pixel) lives in
//    per-thread shared-memory slots, not in registers across the traversal loop;
//  * while-while traversal with a resumable cursor: every lane runs inner-node visits until it holds a leaf,
//    the warp tests the postponed leaves together, and leaves the loop as soon as fewer than `trav_threshold`
//    lanes still traverse (finished lanes never idle until the slowest lane ends);
//  * the inner-node visit is branch-free: three-FMA slab tests on centre/half-extent boxes (FAST; the exact
//    Aabb::hit2 arithmetic otherwise), predicates feeding one predicated push / pop on a sentinel stack;
//  * the Perlin marble is evaluated by the whole warp (coop_turbulence);
//  * per-pixel sums are 64-bit fixed-point shared-memory atomics: the image is bit-deterministic and independent
//    of scheduling, row ranges, tile shards and sample ranges.
// DESIGN.md §3 has the measurements behind each of these.
// ------------------------------------------------------------------------------------------
template <class Acc, bool COUNT, bool FAST, int BLK>
__global__ void __launch_bounds__(BLK, 1) path_trace_kernel_v2(const __grid_constant__ RenderArgs a) {
    extern __shared__ float4 smem[];
    int* stack_base;
    Acc acc = Stager<Acc>::stage(a.scene, a.plan, smem, &stack_base);
    int* stack = stack_base + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt = (1u << lane) - 1u;
    // per-warp fixed-point accumulators [32 pixels][3] behind the stack columns
    long long* wacc = reinterpret_cast<long long*>(stack_base + a.plan.stack_depth * BLK) + (threadIdx.x >> 5) * 96;
    // per-warp queue of generated primary rays, SoA [RAYQ_FIELDS][RAYQ_SLOTS] behind the accumulators
    uint32_t* rayq = reinterpret_cast<uint32_t*>(reinterpret_cast<long long*>(stack_base + a.plan.stack_depth * BLK) + (BLK / 32) * 96)
                     + (threadIdx.x >> 5) * (RAYQ_FIELDS * RAYQ_SLOTS);
    // Per-path state that is touched once per bounce — ray_color's attenuation and emitted accumulators (render.rs:24-25)
    // and the path's tile pixel — lives in shared memory behind the ray queue, SoA [7][BLK]: seven registers fewer across
    // the traversal loop.  `emitted` is only materialised for scenes with emissive materials (it is zero until the path ends
    // otherwise).  Slot k of this thread = ps_s + k * BLK * 4 in the shared window.
    const uint32_t ps_s = (uint32_t)__cvta_generic_to_shared(reinterpret_cast<uint32_t*>(reinterpret_cast<long long*>(stack_base + a.plan.stack_depth * BLK) + (BLK / 32) * 96)
                                                             + (BLK / 32) * (RAYQ_FIELDS * RAYQ_SLOTS) + threadIdx.x);
    auto ps_ld = [&](int k) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(ps_s + (uint32_t)k * BLK * 4u) : "memory"); return v; };
    auto ps_st = [&](int k, float v) { asm volatile("st.shared.f32 [%0], %1;" :: "r"(ps_s + (uint32_t)k * BLK * 4u), "f"(v) : "memory"); };
    auto ps_ld3 = [&](int k) { return f3(ps_ld(k), ps_ld(k + 1), ps_ld(k + 2)); };
    auto ps_st3 = [&](int k, float3 v) { ps_st(k, v.x); ps_st(k + 1, v.y); ps_st(k + 2, v.z); };
    constexpr int PS_ATTEN = 0, PS_EMIT = 3, PS_PIXEL = 6;
    const bool has_emitters = a.scene.has_emitters != 0u;
    const float T_MIN = 0.001f;                      // render.rs:31
    const bool has_perlin = a.scene.perlin != nullptr;
    // (the Perlin tables stay in global memory behind L1: a shared-memory copy reached through generic loads measured 0.4 % slower)
    const PerlinRec* perlin_tables = a.scene.perlin;
    const float sample_lim = 2.0e9f / (float)a.lim_samples;   // acc_add: the fixed-point sum cannot wrap

    unsigned long long w_rays = 0, w_paths = 0, w_exh = 0, w_nodes = 0, w_prims = 0;
    // lane-utilisation diagnostics (COUNT only, lane 0 of each warp):
    //  d0 outer iterations, d1 sum of alive lanes, d2 sum of lanes with no samples left,
    //  d3 traversal rounds, d4 sum of traversing lanes per round, d5 sum of lanes shaded,
    //  d6 sum of lanes regenerated, d7 inner-node visit steps (warp-level)
    unsigned long long d0 = 0, d1 = 0, d2 = 0, d3 = 0, d4 = 0, d5 = 0, d6 = 0, d7 = 0;

    for (;;) {
        unsigned int j = 0, listed = 0;
        if (lane == 0) {
            j = atomicAdd(&a.counters->tile_counter, 1u);
            if (a.tile_list && j < a.chunks * a.my_tiles) listed = a.tile_list[j % a.my_tiles];
        }
        j = __shfl_sync(FULL, j, 0);
        // Work item j = (sample range j / my_tiles, tile j % my_tiles): a tile's samples are split over several warps when the
        // frame has too few tiles to balance the grid (1200x800 at 500 spp is 10.5 whole tiles per warp: the kernel ran 18 %
        // below its rate on frames with 4x the tiles).  Bottom rows first within every range.
        const uint32_t chunk = j / a.my_tiles;
        if (chunk >= a.chunks) break;
        uint32_t t = (j - chunk * a.my_tiles) * a.shard_count + a.shard_index;
        if (a.tile_list) t = __shfl_sync(FULL, listed, 0);
        const uint32_t s_begin = a.chunk_begin[chunk];
        const uint32_t s_count = a.chunk_begin[chunk + 1u] - s_begin;
        uint32_t ty = t / a.tiles_x, tx = t - ty * a.tiles_x;
        const uint32_t px0 = tx * TILE_W, py0 = (a.tile_row0 + ty) * TILE_H;
        const uint32_t my_px = px0 + (lane & (TILE_W - 1)), my_py = py0 + (lane >> 3);
        const bool valid = my_px < a.cam.width && my_py >= a.row_begin && my_py < a.row_end;
        // The tile's work list: item i = sample * nv + k (k-th valid pixel).  Any lane takes the
        // next item when its path ends, so all lanes stay busy until the tile is finished
        // (with lane = pixel, 17 % of the lanes sat out of samples at tile ends).
        const unsigned valid_mask = __ballot_sync(FULL, valid);
        const uint32_t nv = (uint32_t)__popc(valid_mask);
        const uint32_t n_items = s_count * nv;
        uint32_t next_item = 0;          // next work-list item to generate
        uint32_t q_head = 0, q_count = 0;  // the warp's ring of generated primary rays
        for (int k = lane; k < 96; k += 32) wacc[k] = 0;
        __syncwarp();
        uint32_t nrays = 0, nexh = 0;   // nrays: warp total (same value in every lane), nexh: per lane
        TravCounters tc; tc.nodes = 0; tc.prims = 0;
        Rng rng; rng.state = 0; rng.inc = 1;
        RayF ray = make_ray_shade(f3(0, 0, 0), f3(0, 0, 1));
        uint32_t depth = 0;
        int node = B200RT_TRAV_DONE;
        const uint32_t stack_s = (uint32_t)__cvta_generic_to_shared(stack);
        uint32_t top_sp = stack_s + BLK * 4;   // shared-window address of the next free slot of this lane's stack column
        Closest c; c.t = INFINITY; c.code = -1;
        stack[0] = B200RT_TRAV_DONE;     // sentinel: popping it ends a traversal (trav_inner_s)

        // One outer iteration = shade the lanes whose traversal finished, hand new paths to the
        // lanes without one, set up the new segments of BOTH groups together (one copy of the ray
        // set-up + up-front primitive code, run at ~30 lanes instead of twice at 6 and 18), traverse.
        for (;;) {
            // ---- shade: ray_color's loop body, render.rs:31-46 ----
            bool fin = depth != 0u && node == B200RT_TRAV_DONE;     // a lane holds a path while depth != 0
            if (COUNT) { d0 += 1; d5 += __popc(__ballot_sync(FULL, fin)); }
            bool hit = fin && c.code >= 0;
            bool done = false, setup = false;
            HitRec h;
            ShadePrep sp_;
            sp_.tex.need_perlin = false; sp_.tex.perlin_idx = 0;
            h.p = f3(0.f, 0.f, 0.f);
            float3 radiance = f3(0.f, 0.f, 0.f);         // what the path adds to its pixel when it ends in this iteration
            if (fin && !hit) {                           // render.rs:44-45: emitted + attenuation * background
                const float3 bg = background(a.scene, ray.d);
                // (`emitted` is loaded before `attenuation` in both updates, the order of the code before the explicit fmaf)
                if (has_emitters) { const float3 e = ps_ld3(PS_EMIT); radiance = fma_f3(ps_ld3(PS_ATTEN), bg, e); }
                else radiance = mul_rn3(ps_ld3(PS_ATTEN), bg);
                done = true;
            }
            if (hit) {
                h = make_hit(ray, acc, c);
                sp_ = shade_prepare(a.scene, acc, h);
            }
            float turb = 0.0f;
            if (has_perlin && __any_sync(FULL, hit && sp_.tex.need_perlin))   // warp-uniform: skip the call when no lane asks
                turb = coop_turbulence(perlin_tables, hit && sp_.tex.need_perlin, h.p, sp_.tex.perlin_idx);
            if (hit) {
                float3 albedo = sp_.tex.need_perlin ? marble(sp_.tex.perlin_scale, h.p, turb) : sp_.tex.rgb;
                ShadeOut so = shade_finish(ray, h, sp_.m, albedo, rng);
                if (so.has_emission) {                   // only scenes with emitters get here
                    const float3 e = ps_ld3(PS_EMIT);
                    ps_st3(PS_EMIT, fma_f3(ps_ld3(PS_ATTEN), so.emission, e));
                }
                done = !so.scattered;
                if (!done) {
                    if (--depth == 0) { done = true; ++nexh; }
                    else {
                        ray.o = so.o; ray.d = so.d; setup = true;
                        if (so.has_mul) ps_st3(PS_ATTEN, mul_rn3(ps_ld3(PS_ATTEN), so.mul));
                    }
                }
            }
            if (done) {
                if (has_emitters && hit) radiance = ps_ld3(PS_EMIT);      // ended on a light or ran out of depth: `emitted` so far
                acc_add(wacc, __float_as_uint(ps_ld(PS_PIXEL)), radiance, sample_lim);
                depth = 0;
            }

            // ---- path regeneration: render_scanline's sample loop, render.rs:60-66 ----
            // Primary rays are generated 32 at a time into the warp's queue (all lanes busy: RNG
            // keying, jitter, lens rejection loop, Camera::pixel_ray) and handed out to the ~6 lanes
            // per iteration whose path ended; generating them on demand ran that code at 6 lanes.
            unsigned want_m = __ballot_sync(FULL, depth == 0u);
            if ((uint32_t)__popc(want_m) < a.regen_min) want_m = 0u;      // too few free lanes: they wait an iteration
            const uint32_t want = (uint32_t)__popc(want_m);
            if (q_count < want && next_item < n_items) {           // warp-uniform
                __syncwarp();
                // top the ring up to 32 entries: the first (32 - q_count) lanes generate
                const uint32_t n_new = min(RAYQ_SLOTS - q_count, n_items - next_item);
                uint32_t item = next_item + (uint32_t)lane;
                if ((uint32_t)lane < n_new) {
                    uint32_t sidx = (nv == 32u) ? (item >> 5) : item / nv;
                    uint32_t kth = item - sidx * nv;
                    uint32_t qpl = (nv == 32u) ? kth : (uint32_t)__fns(valid_mask, 0, (int)kth + 1);
                    uint32_t px = px0 + (qpl & (TILE_W - 1)), py = py0 + (qpl >> 3);
                    Rng qr;
                    qr.init(a.keys, py * a.cam.width + px, a.sample_offset + s_begin + sidx);
                    float jx = (float)px + qr.gen();
                    float jy = (float)py + qr.gen();
                    float3 qo, qd;
                    pixel_ray(a.cam, qr, jx, jy, &qo, &qd);
                    uint32_t slot = (q_head + q_count + (uint32_t)lane) & (RAYQ_SLOTS - 1);
                    rayq[0 * RAYQ_SLOTS + slot] = __float_as_uint(qo.x); rayq[1 * RAYQ_SLOTS + slot] = __float_as_uint(qo.y);
                    rayq[2 * RAYQ_SLOTS + slot] = __float_as_uint(qo.z); rayq[3 * RAYQ_SLOTS + slot] = __float_as_uint(qd.x);
                    rayq[4 * RAYQ_SLOTS + slot] = __float_as_uint(qd.y); rayq[5 * RAYQ_SLOTS + slot] = __float_as_uint(qd.z);
                    rayq[6 * RAYQ_SLOTS + slot] = qr.state; rayq[7 * RAYQ_SLOTS + slot] = qr.inc; rayq[8 * RAYQ_SLOTS + slot] = qpl;
                }
                next_item += n_new; q_count += n_new;
                __syncwarp();
            }
            const uint32_t rank = (uint32_t)__popc(want_m & lt);
            bool regen = depth == 0u && ((want_m >> lane) & 1u) && rank < q_count;
            if (COUNT) { d6 += __popc(__ballot_sync(FULL, regen)); d2 += __popc(__ballot_sync(FULL, depth == 0u && !regen)); }
            if (regen) {
                uint32_t slot = (q_head + rank) & (RAYQ_SLOTS - 1);
                ray.o = f3(__uint_as_float(rayq[0 * RAYQ_SLOTS + slot]), __uint_as_float(rayq[1 * RAYQ_SLOTS + slot]), __uint_as_float(rayq[2 * RAYQ_SLOTS + slot]));
                ray.d = f3(__uint_as_float(rayq[3 * RAYQ_SLOTS + slot]), __uint_as_float(rayq[4 * RAYQ_SLOTS + slot]), __uint_as_float(rayq[5 * RAYQ_SLOTS + slot]));
                rng.state = rayq[6 * RAYQ_SLOTS + slot]; rng.inc = rayq[7 * RAYQ_SLOTS + slot];
                ps_st(PS_PIXEL, __uint_as_float(rayq[8 * RAYQ_SLOTS + slot]));
                ps_st3(PS_ATTEN, f3(1, 1, 1));
                if (has_emitters) ps_st3(PS_EMIT, f3(0, 0, 0));
                depth = a.max_depth;
                setup = depth != 0u;
            }
            {
                uint32_t taken = min(want, q_count);
                q_head = (q_head + taken) & (RAYQ_SLOTS - 1); q_count -= taken;
            }
            if (!__any_sync(FULL, depth != 0u)) break;
            if (COUNT) d1 += __popc(__ballot_sync(FULL, depth != 0u));

            // ---- new segment: per-ray constants, then the scene-spanning primitives ----
            if (setup) {
                // IEEE reciprocals, taken once: the up-front rect/box tests need exactly these
                // (bit-reproducible on the CPU), and the slab tests take them too
                float3 inv_e = f3(__frcp_rn(ray.d.x), __frcp_rn(ray.d.y), __frcp_rn(ray.d.z));
                ray.inv = FAST ? f3(clamp_inv(inv_e.x), clamp_inv(inv_e.y), clamp_inv(inv_e.z)) : inv_e;
                ray.nood = f3(-(ray.o.x * ray.inv.x), -(ray.o.y * ray.inv.y), -(ray.o.z * ray.inv.z));
                c.t = INFINITY; c.code = -1;
                // the list is indexed in the kernel parameters (constant bank): a register copy indexed by a
                // loop counter would live in local memory
#pragma unroll 1
                for (uint32_t k = 0; k < a.scene.n_top_prims; ++k) {
                    if (COUNT) tc.prims++;
                    hit_leaf(ray, acc, a.scene.top_prims[k], T_MIN, c, &inv_e);
                }
                node = 0; top_sp = stack_s + BLK * 4;
            }
            nrays += (uint32_t)__popc(__ballot_sync(FULL, setup));   // warp-uniform count: no per-lane counter to keep live

            // ---- traversal: BboxTree::hit_workspace, bvh/bbox_tree.rs:56-91 ----
            for (;;) {
                if (COUNT) { d3 += 1; d4 += __popc(__ballot_sync(FULL, node != B200RT_TRAV_DONE)); }
                // (a warp-uniform inner loop that stops below a lane threshold, and a cap on the steps per
                //  round, were measured: 15-18 lanes per step instead of 13.6, but no faster — profiles/README.md)
                while (node >= 0 && node != B200RT_TRAV_DONE) {
                    if (COUNT) d7 += (__ffs(__activemask()) - 1 == lane) ? 1 : 0;
                    trav_inner_s<COUNT, FAST>(ray, acc, top_sp, BLK * 4, T_MIN, c, node, tc);
                }
                if (node < 0) trav_leaf_s<COUNT>(ray, acc, top_sp, BLK * 4, T_MIN, c, node, tc);
                unsigned still = __ballot_sync(FULL, node != B200RT_TRAV_DONE);
                if ((uint32_t)__popc(still) < a.trav_threshold) break;
            }
        }
        __syncwarp();
        if (valid) {
            if (a.fix) {
                // several warps (or passes) hold partial sums of this pixel: exact 64-bit integer adds in global memory (native RED.ADD.64),
                // so the total — and the float finalize_kernel derives from it — is the same whatever the split or the order
                unsigned long long* f = reinterpret_cast<unsigned long long*>(a.fix) + ((size_t)my_py * a.cam.width + my_px) * 3;
                atomicAdd(f + 0, (unsigned long long)wacc[lane * 3 + 0]);
                atomicAdd(f + 1, (unsigned long long)wacc[lane * 3 + 1]);
                atomicAdd(f + 2, (unsigned long long)wacc[lane * 3 + 2]);
            } else {
                const float inv = 1.0f / 4294967296.0f;
                float4* dst = a.accum + (my_py * a.cam.width + my_px);
                float4 v = make_float4((float)wacc[lane * 3 + 0] * inv, (float)wacc[lane * 3 + 1] * inv, (float)wacc[lane * 3 + 2] * inv, (float)a.samples);
                if (a.accumulate) { float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
                *dst = v;
            }
        }
        __syncwarp();
        w_rays += lane == 0 ? nrays : 0u; w_exh += nexh; w_paths += lane == 0 ? n_items : 0u;   // every work-list item became one path
        if (COUNT) { w_nodes += tc.nodes; w_prims += tc.prims; }
    }
    for (int o = 16; o > 0; o >>= 1) {
        w_rays += __shfl_down_sync(FULL, w_rays, o);
        w_paths += __shfl_down_sync(FULL, w_paths, o);
        w_exh += __shfl_down_sync(FULL, w_exh, o);
        if (COUNT) { w_nodes += __shfl_down_sync(FULL, w_nodes, o); w_prims += __shfl_down_sync(FULL, w_prims, o); }
    }
    if (lane == 0) {
        atomicAdd(&a.counters->rays, w_rays);
        atomicAdd(&a.counters->paths, w_paths);
        atomicAdd(&a.counters->exhausted, w_exh);
        if (COUNT) { atomicAdd(&a.counters->nodes, w_nodes); atomicAdd(&a.counters->prims, w_prims); }
    }
    if (COUNT) {
        // d7 was counted by whichever lane led each divergent step: sum it over the warp
        for (int o = 16; o > 0; o >>= 1) d7 += __shfl_down_sync(FULL, d7, o);
        if (lane == 0) {
            atomicAdd(&a.counters->diag[0], d0); atomicAdd(&a.counters->diag[1], d1); atomicAdd(&a.counters->diag[2], d2); atomicAdd(&a.counters->diag[3], d3);
            atomicAdd(&a.counters->diag[4], d4); atomicAdd(&a.counters->diag[5], d5); atomicAdd(&a.counters->diag[6], d6); atomicAdd(&a.counters->diag[7], d7);
        }
    }
}


// chunks > 1: fixed-point sums -> the float4 accumulation buffer, for exactly the pixels the launch rendered
// (same arithmetic as the kernel's own tile write-back, so the result does not depend on `chunks`).
__global__ void finalize_kernel(const __grid_constant__ RenderArgs a) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = a.row_begin + blockIdx.y;
    if (x >= a.cam.width || y >= a.row_end) return;
    const uint32_t t = (y / TILE_H - a.tile_row0) * a.tiles_x + x / TILE_W;
    if (t % a.shard_count != a.shard_index) return;
    const size_t p = (size_t)y * a.cam.width + x;
    const float inv = 1.0f / 4294967296.0f;
    float4 v = make_float4((float)a.fix[p * 3 + 0] * inv, (float)a.fix[p * 3 + 1] * inv, (float)a.fix[p * 3 + 2] * inv, (float)a.samples);
    if (a.accumulate) { float4 o = a.accum[p]; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
    a.accum[p] = v;
}

// ------------------------------------------------------------------------------------------
// Tile-adaptive sampling (b200rt_render_adaptive).  After pass k >= 1 the pass buffer P holds the sums of the samples
// [n, n + s) of every active tile and F those of [0, n).  One warp per active tile, one lane per pixel: e_p from the two
// independent means (adaptive_plan.hpp), e_T = the warp maximum; P is added into F exactly (64-bit integers) and zeroed for the
// next pass; a tile that stops writes its float4 pixels with finalize_kernel's arithmetic, so they equal a plain render of
// n + s samples bit for bit.
// ------------------------------------------------------------------------------------------
struct MergeArgs {
    const uint32_t* list;       // the active tiles (NULL: all tiles 0 .. n_active)
    uint32_t n_active;
    long long* F;               // [H][W][3] sums before the pass
    long long* P;               // [H][W][3] sums of the pass
    float4* accum;
    float* tile_error;          // per tile of the grid covering [row_begin, row_end): e_T at its last pass
    uint32_t* keep;             // per list entry: 1 = still active
    uint32_t n, s;              // samples before the pass, samples of the pass
    uint32_t last;              // n + s == max_samples: every tile stops
    float threshold;
    uint32_t W, row_begin, row_end, tiles_x, tile_row0;
};

__global__ void adaptive_merge_kernel(const __grid_constant__ MergeArgs a) {
    const uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t lane = threadIdx.x & 31u;
    if (i >= a.n_active) return;                 // warp-uniform
    const uint32_t t = a.list ? a.list[i] : i;
    const uint32_t ty = t / a.tiles_x, tx = t - ty * a.tiles_x;
    const uint32_t x = tx * TILE_W + (lane & (TILE_W - 1)), y = (a.tile_row0 + ty) * TILE_H + (lane >> 3);
    const bool valid = x < a.W && y >= a.row_begin && y < a.row_end;
    const size_t p = ((size_t)y * a.W + x) * 3;
    float e = 0.0f;
    long long sum[3] = {0, 0, 0};
    if (valid) {
        const long long f[3] = {a.F[p], a.F[p + 1], a.F[p + 2]};
        const long long q[3] = {a.P[p], a.P[p + 1], a.P[p + 2]};
        e = adaptive_pixel_error(f, q, a.n, a.s);
        for (int c = 0; c < 3; ++c) { sum[c] = f[c] + q[c]; a.F[p + c] = sum[c]; a.P[p + c] = 0; }
    }
    for (int o = 16; o > 0; o >>= 1) e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, o));
    const bool stop = a.last != 0u || e <= a.threshold;
    if (valid && stop) {
        const float inv = 1.0f / 4294967296.0f;
        a.accum[p / 3] = make_float4((float)sum[0] * inv, (float)sum[1] * inv, (float)sum[2] * inv, (float)(a.n + a.s));
    }
    if (lane == 0) { a.tile_error[t] = e; a.keep[i] = stop ? 0u : 1u; }
}

// The next pass's tile list: the entries of `list` (NULL: 0 .. n) whose keep flag is set, in ascending order, so that the next
// pass still schedules bottom rows first and is the same run to run.  One CTA: a few hundred thousand flags at most.
constexpr int COMPACT_THREADS = 1024;
__global__ void __launch_bounds__(COMPACT_THREADS) adaptive_compact_kernel(const uint32_t* list, const uint32_t* keep, uint32_t n,
                                                                            uint32_t* out, uint32_t* out_count) {
    __shared__ uint32_t warp_counts[COMPACT_THREADS / 32];
    __shared__ uint32_t base;
    const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (uint32_t i0 = 0; i0 < n; i0 += COMPACT_THREADS) {
        const uint32_t i = i0 + threadIdx.x;
        const bool k = i < n && keep[i] != 0u;
        const unsigned m = __ballot_sync(0xffffffffu, k);
        if (lane == 0) warp_counts[w] = (uint32_t)__popc(m);
        __syncthreads();
        uint32_t at = base;
        for (uint32_t v = 0; v < w; ++v) at += warp_counts[v];
        if (k) out[at + (uint32_t)__popc(m & ((1u << lane) - 1u))] = list ? list[i] : i;
        __syncthreads();
        if (threadIdx.x == 0) { uint32_t total = 0; for (uint32_t v = 0; v < COMPACT_THREADS / 32; ++v) total += warp_counts[v]; base += total; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *out_count = base;
}

}  // namespace b200rt
