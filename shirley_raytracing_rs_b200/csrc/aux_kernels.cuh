// aux_kernels.cuh — K1 closest-hit batch, K3 resolve (+ the fused cross-GPU form and its flag barrier), K4 parity hooks, the FFMA-chain microbenchmark
// (included by b200rt.cu; everything lives in namespace b200rt)
#pragma once
#include "render_kernel.cuh"

namespace b200rt {

// ------------------------------------------------------------------------------------------
// K1: closest-hit over a ray array, one thread per ray (grid-stride).
// ------------------------------------------------------------------------------------------
struct HitArgs {
    DeviceScene scene; SmemPlan plan;
    const B200rtRay* rays; size_t n; float t_min, t_max;
    int32_t* ids; B200rtHit* hits; Counters* counters;
    unsigned long long* next_ray;      // the global ray counter the persistent warps draw from
};

// K1 runs the SAME traversal code as the render kernel (per-segment set-up with shared IEEE reciprocals, up-front
// primitives, trav_inner_s / trav_leaf_s over the sentinel stack; FAST = centre/half-extent boxes) so that the
// bit-exact id / t / normal parity tests exercise the product's traversal, not a parity-only twin.
// Like the render kernel it is persistent and refills lanes: a warp takes rays from a global counter, every lane
// traverses until it holds a leaf, the held leaves are tested together, and as soon as fewer than `refill` lanes
// still traverse, the finished lanes store their results and take new rays (one thread per ray and a loop until the
// warp's slowest ray ends ran at 129-314 Mrays/s on the criterion-shaped lattice: the lanes idled).
template <class Acc, bool COUNT, bool FAST>
__global__ void __launch_bounds__(BLOCK) closest_hit_kernel(const __grid_constant__ HitArgs a) {
    extern __shared__ float4 smem[];
    int* stack_base;
    Acc acc = Stager<Acc>::stage(a.scene, a.plan, smem, &stack_base);
    int* stack = stack_base + threadIdx.x;
    stack[0] = B200RT_TRAV_DONE;
    const uint32_t stack_s = (uint32_t)__cvta_generic_to_shared(stack);
    const int lane = threadIdx.x & 31;
    const unsigned FULL = 0xffffffffu;
    const unsigned lt = (1u << lane) - 1u;
    const uint32_t refill = 12;                         // leave the traversal loop below this many traversing lanes
    TravCounters tc; tc.nodes = 0; tc.prims = 0;
    unsigned long long nr = 0;
    long long mine = -1;                                // index of the ray this lane holds, -1 = none
    bool exhausted = false;                             // warp-uniform: the ray counter ran past the array
    RayF ray = make_ray_shade(f3(0, 0, 0), f3(0, 0, 1));
    Closest c; c.t = a.t_max; c.code = -1;
    int node = B200RT_TRAV_DONE;
    uint32_t top_sp = stack_s + BLOCK * 4;
    for (;;) {
        // ---- store finished rays ----
        if (mine >= 0 && node == B200RT_TRAV_DONE) {
            ++nr;
            int id = c.code < 0 ? -1 : (int)((uint32_t)c.code & B200RT_CODE_ID_MASK);
            a.ids[mine] = id;
            if (a.hits) {
                B200rtHit out;
                memset(&out, 0, sizeof out);
                out.id = id;
                if (id >= 0) {
                    HitRec h = make_hit(ray, acc, c);
                    float u, v;
                    hit_uv(h, acc, &u, &v);
                    out.t = h.t; out.p[0] = h.p.x; out.p[1] = h.p.y; out.p[2] = h.p.z;
                    out.n[0] = h.n.x; out.n[1] = h.n.y; out.n[2] = h.n.z;
                    out.u = u; out.v = v; out.front_face = h.front ? 1 : 0;
                }
                a.hits[mine] = out;
            }
            mine = -1;
        }
        // ---- refill: the free lanes take the next rays ----
        const unsigned want_m = __ballot_sync(FULL, mine < 0);
        if (want_m && !exhausted) {
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(a.next_ray, (unsigned long long)__popc(want_m));
            base = __shfl_sync(FULL, base, 0);
            if (base >= a.n) exhausted = true;
            const unsigned long long i = base + (unsigned long long)__popc(want_m & lt);
            if (mine < 0 && i < a.n) {
                mine = (long long)i;
                B200rtRay in = a.rays[i];
                ray.o = f3(in.ox, in.oy, in.oz); ray.d = f3(in.dx, in.dy, in.dz);
                float3 inv_e = f3(__frcp_rn(ray.d.x), __frcp_rn(ray.d.y), __frcp_rn(ray.d.z));
                ray.inv = FAST ? f3(clamp_inv(inv_e.x), clamp_inv(inv_e.y), clamp_inv(inv_e.z)) : inv_e;
                ray.nood = f3(-(ray.o.x * ray.inv.x), -(ray.o.y * ray.inv.y), -(ray.o.z * ray.inv.z));
                c.t = a.t_max; c.code = -1;
#pragma unroll 1
                for (uint32_t k = 0; k < a.scene.n_top_prims; ++k) {
                    if (COUNT) tc.prims++;
                    hit_leaf(ray, acc, a.scene.top_prims[k], a.t_min, c, &inv_e);
                }
                node = 0; top_sp = stack_s + BLOCK * 4;
            }
        }
        if (!__any_sync(FULL, mine >= 0)) break;
        // ---- traverse ----
        for (;;) {
            while (node >= 0 && node != B200RT_TRAV_DONE) trav_inner_s<COUNT, FAST>(ray, acc, top_sp, BLOCK * 4, a.t_min, c, node, tc);
            if (node < 0) trav_leaf_s<COUNT>(ray, acc, top_sp, BLOCK * 4, a.t_min, c, node, tc);
            const unsigned still = __ballot_sync(FULL, node != B200RT_TRAV_DONE);
            if ((uint32_t)__popc(still) < (exhausted ? 1u : refill)) break;
        }
    }
    if (a.counters) {
        atomicAdd(&a.counters->rays, nr);
        if (COUNT) { atomicAdd(&a.counters->nodes, (unsigned long long)tc.nodes); atomicAdd(&a.counters->prims, (unsigned long long)tc.prims); }
    }
}

// ------------------------------------------------------------------------------------------
// K3: resolve.  to_image (image.rs:34-40): c * (1/samples), sqrt, (x * 255.999) as u8
// (saturating, NaN -> 0), vertical flip.  Evaluated in f64 like the reference so the bytes
// are bit-identical to the oracle's for the same accumulation buffer.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned char to_pixel(double x) {
    double v = x * 255.999;
    if (!(v > 0.0)) return 0;
    if (v >= 255.0) return 255;
    return (unsigned char)v;
}
__global__ void resolve_kernel(const float4* __restrict__ accum, uint32_t W, uint32_t H, uint32_t samples, uint8_t* __restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t j = blockIdx.y;
    if (i >= W || j >= H) return;
    float4 c = accum[(size_t)j * W + i];
    double n = samples ? (double)samples : (double)c.w;
    double inv = 1.0 / n;
    uint8_t* px = out + ((size_t)(H - 1 - j) * W + i) * 3;
    px[0] = to_pixel(sqrt((double)c.x * inv));
    px[1] = to_pixel(sqrt((double)c.y * inv));
    px[2] = to_pixel(sqrt((double)c.z * inv));
}


// K3p: the cross-GPU sum fused into the resolve (SURVEY.md §2 K3).  With sample-range sharding
// every GPU holds a full-frame float4 buffer of its own samples; instead of an NCCL reduce onto
// one GPU followed by resolve_kernel there, each GPU takes a band of rows, reads that band from
// EVERY GPU's buffer through NVLink peer pointers (coalesced 16-byte loads), adds them in rank
// order (so the bytes do not depend on timing), applies to_image's arithmetic and stores the
// RGB8 band — through a peer pointer again — into the frame on the root GPU.  One pass, no
// intermediate reduced buffer, and the traffic is spread over all GPUs' links.
constexpr int MAX_PEERS = 16;
struct PeerResolveArgs {
    const float4* accum[MAX_PEERS];
    uint32_t n_peers, W, H, samples, row_begin, row_end;
    uint8_t* out;
    const uint32_t* abort_flag;     // non-zero (a flag wait timed out: some peer's buffer is not complete) -> store nothing
};
__device__ __forceinline__ float4 peer_sum(const PeerResolveArgs& a, size_t idx) {
    float4 c = __ldcg(a.accum[0] + idx);        // .cg: peer data must not be served from a stale L1 line
    for (uint32_t r = 1; r < a.n_peers; ++r) {
        float4 v = __ldcg(a.accum[r] + idx);
        c.x += v.x; c.y += v.y; c.z += v.z; c.w += v.w;
    }
    return c;
}
__global__ void resolve_peers_kernel(const __grid_constant__ PeerResolveArgs a) {
    const uint32_t j = a.row_begin + blockIdx.y;
    if (j >= a.row_end) return;
    if (a.abort_flag && *reinterpret_cast<const volatile uint32_t*>(a.abort_flag) != 0u) return;   // never resolve an incomplete frame
    const uint32_t groups = (a.W + 3) / 4;
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= groups) return;
    const uint32_t i0 = g * 4;
    uint8_t bytes[12];
    uint32_t n_px = min(4u, a.W - i0);
    for (uint32_t k = 0; k < n_px; ++k) {
        float4 c = peer_sum(a, (size_t)j * a.W + i0 + k);
        double n = a.samples ? (double)a.samples : (double)c.w;
        double inv = 1.0 / n;
        bytes[3 * k + 0] = to_pixel(sqrt((double)c.x * inv));
        bytes[3 * k + 1] = to_pixel(sqrt((double)c.y * inv));
        bytes[3 * k + 2] = to_pixel(sqrt((double)c.z * inv));
    }
    uint8_t* px = a.out + ((size_t)(a.H - 1 - j) * a.W + i0) * 3;
    if (n_px == 4 && ((uintptr_t)px & 3u) == 0) {
        uint32_t* w = reinterpret_cast<uint32_t*>(px);
        w[0] = bytes[0] | (bytes[1] << 8) | (bytes[2] << 16) | ((uint32_t)bytes[3] << 24);
        w[1] = bytes[4] | (bytes[5] << 8) | (bytes[6] << 16) | ((uint32_t)bytes[7] << 24);
        w[2] = bytes[8] | (bytes[9] << 8) | (bytes[10] << 16) | ((uint32_t)bytes[11] << 24);
    } else {
        for (uint32_t k = 0; k < 3 * n_px; ++k) px[k] = bytes[k];
    }
}


// Cross-GPU ordering for the fused resolve without a library collective: every rank owns a small flag
// array in peer-visible memory, [slot][rank] epochs.  signal = "my stream has reached this point" written
// into every peer's array (release, system scope); wait = spin until all peers' epochs arrived (acquire).
// slot 0 = "my accumulation buffer is complete", slot 1 = "I am done reading your buffer".
constexpr uint32_t PEER_FLAG_STRIDE = 16;
struct PeerSignalArgs { uint32_t* flags[MAX_PEERS]; uint32_t n_peers, my_rank, slot, epoch; };
__global__ void peer_signal_kernel(const __grid_constant__ PeerSignalArgs a) {
    uint32_t p = threadIdx.x;
    if (p >= a.n_peers) return;
    __threadfence_system();
    uint32_t* dst = a.flags[p] + a.slot * PEER_FLAG_STRIDE + a.my_rank;
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(dst), "r"(a.epoch) : "memory");
}
__global__ void peer_wait_kernel(const uint32_t* my_flags, uint32_t n_peers, uint32_t slot, uint32_t epoch, unsigned long long timeout_ns, uint32_t* timed_out) {
    uint32_t r = threadIdx.x;
    if (r >= n_peers) return;
    const uint32_t* src = my_flags + slot * PEER_FLAG_STRIDE + r;
    unsigned long long t0; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (;;) {
        uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
        if ((int32_t)(v - epoch) >= 0) break;
        unsigned long long t1; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        // a missing peer must not hang the GPU: record it (the fused resolve that follows sees the word and stores
        // nothing; the host reads it with b200rt_peer_timed_out and fails the frame) and let the stream go on
        if (t1 - t0 > timeout_ns) { atomicExch(timed_out, 1u + r); __threadfence(); break; }
        __nanosleep(200);
    }
}

// ------------------------------------------------------------------------------------------
// parity-hook kernels
// ------------------------------------------------------------------------------------------
__global__ void aabb_hit_kernel(const float* __restrict__ boxes6, const B200rtRay* __restrict__ rays, size_t n, float t_min, float t_max, uint8_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    B200rtRay in = rays[i];
    RayF ray = make_ray(f3(in.ox, in.oy, in.oz), f3(in.dx, in.dy, in.dz));
    const float* b = boxes6 + i * 6;
    float e;
    out[i] = aabb_hit2(ray, b[0], b[1], b[2], b[3], b[4], b[5], t_min, t_max, &e) ? 1 : 0;
}

// The hooks' random stream of record i: b200rt_rng(seed, i, 0), or with `stream` (three words per record) b200rt_rng(seed, a, b)
// after `skip` draws, which continues a render's path stream (pixel, sample) where the render is.
__device__ __forceinline__ Rng hook_rng(RngKeys keys, const uint32_t* stream, size_t i) {
    Rng rng;
    if (!stream) { rng.init(keys, (uint32_t)i, 0u); return rng; }
    rng.init(keys, stream[3 * i], stream[3 * i + 1]);
    for (uint32_t k = stream[3 * i + 2]; k != 0u; --k) rng.state = rng.state * 747796405u + rng.inc;
    return rng;
}
// draws taken since the state was s0 = LCG steps from s0 to rng.state, recounted by stepping
__device__ __forceinline__ uint32_t draws_since(uint32_t s0, const Rng& rng) {
    uint32_t st = s0, k = 0;
    while (st != rng.state && k < 4096) { st = st * 747796405u + rng.inc; ++k; }
    return k;
}

struct ScatterArgs { DeviceScene scene; const B200rtRay* rays; const B200rtHit* hits; size_t n; RngKeys keys; const uint32_t* stream; B200rtScatter* out; };
__global__ void scatter_kernel(const __grid_constant__ ScatterArgs a) {
    // The render kernel's own shading sequence: shade_prepare -> warp-cooperative Perlin -> shade_finish.
    // No early return: coop_turbulence is a warp collective (the grid is rounded up to whole warps).
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = i < a.n;
    GmemAcc acc;
    acc.nodes = reinterpret_cast<const float4*>(a.scene.nodes); acc.geom = reinterpret_cast<const float4*>(a.scene.geom);
    acc.mats = reinterpret_cast<const float4*>(a.scene.mats); acc.tex = reinterpret_cast<const float4*>(a.scene.tex);
    B200rtRay in{}; B200rtHit hi{}; hi.id = -1;
    if (in_range) { in = a.rays[i]; hi = a.hits[i]; }
    B200rtScatter out; memset(&out, 0, sizeof out);
    const bool valid = in_range && hi.id >= 0 && (uint32_t)hi.id < a.scene.n_prims;
    RayF ray = make_ray(f3(in.ox, in.oy, in.oz), f3(in.dx, in.dy, in.dz));
    // rebuild the device hit record from the caller's record; u,v come from the geometry
    HitRec h;
    h.id = hi.id; h.t = hi.t; h.p = f3(hi.p[0], hi.p[1], hi.p[2]); h.n = f3(hi.n[0], hi.n[1], hi.n[2]);
    h.front = hi.front_face != 0;
    h.n_out = h.front ? h.n : -h.n;
    h.type = 0xffu; h.face = 0;
    h.has_uv = true; h.uv_u = hi.u; h.uv_v = hi.v;   // Texture::value(record.u, record.v, ..), lambertian.rs:34
    ShadePrep sp; sp.tex.need_perlin = false; sp.tex.perlin_idx = 0; sp.tex.perlin_scale = 0.f; sp.tex.rgb = f3(0, 0, 0);
    if (valid) sp = shade_prepare(a.scene, acc, h);
    const bool need = valid && sp.tex.need_perlin;
    float turb = 0.0f;
    if (a.scene.perlin != nullptr && __any_sync(0xffffffffu, need)) turb = coop_turbulence(a.scene.perlin, need, h.p, sp.tex.perlin_idx);
    if (valid) {
        Rng rng = hook_rng(a.keys, a.stream, i);
        uint32_t s0 = rng.state;
        float3 atten = f3(1, 1, 1), emit = f3(0, 0, 0);
        float3 albedo = sp.tex.need_perlin ? marble(sp.tex.perlin_scale, h.p, turb) : sp.tex.rgb;
        ShadeOut so = shade_finish(ray, h, sp.m, albedo, rng);
        if (so.has_emission) emit = emit + atten * so.emission;
        if (so.has_mul) atten = atten * so.mul;
        out.ray.ox = so.o.x; out.ray.oy = so.o.y; out.ray.oz = so.o.z;
        out.ray.dx = so.d.x; out.ray.dy = so.d.y; out.ray.dz = so.d.z;
        out.attenuation[0] = atten.x; out.attenuation[1] = atten.y; out.attenuation[2] = atten.z;
        out.emitted[0] = emit.x; out.emitted[1] = emit.y; out.emitted[2] = emit.z;
        out.scattered = so.scattered ? 1 : 0;
        out.draws = draws_since(s0, rng);
    } else if (in_range && hi.id == -1) {        // a miss: the render kernel's background for the ray's direction
        const float3 bg = background(a.scene, ray.d);
        out.emitted[0] = bg.x; out.emitted[1] = bg.y; out.emitted[2] = bg.z;
    }
    if (in_range) a.out[i] = out;
}

__global__ void camera_rays_kernel(DeviceCamera cam, const float* __restrict__ xy, size_t n, RngKeys keys, const uint32_t* stream,
                                   B200rtRay* out, uint32_t* draws) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Rng rng = hook_rng(keys, stream, i);
    const uint32_t s0 = rng.state;
    float3 o, d;
    pixel_ray(cam, rng, xy[2 * i], xy[2 * i + 1], &o, &d);
    B200rtRay r; r.ox = o.x; r.oy = o.y; r.oz = o.z; r.dx = d.x; r.dy = d.y; r.dz = d.z;
    out[i] = r;
    if (draws) draws[i] = draws_since(s0, rng);
}

struct TexArgs { DeviceScene scene; int32_t tex; const float* uvp5; size_t n; float* out; };
__global__ void texture_value_kernel(const __grid_constant__ TexArgs a) {
    // Texture::value the way the render kernel evaluates it: descent per lane, marble turbulence by the whole warp.
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool in_range = i < a.n;
    GmemAcc acc;
    acc.nodes = reinterpret_cast<const float4*>(a.scene.nodes); acc.geom = reinterpret_cast<const float4*>(a.scene.geom);
    acc.mats = reinterpret_cast<const float4*>(a.scene.mats); acc.tex = reinterpret_cast<const float4*>(a.scene.tex);
    const float* q = a.uvp5 + (in_range ? i : 0) * 5;
    HitRec h;
    h.id = -1; h.type = 0xffu; h.face = 0; h.t = 0; h.front = true;
    h.p = f3(q[2], q[3], q[4]); h.n = f3(0, 1, 0); h.n_out = h.n;
    h.has_uv = true; h.uv_u = q[0]; h.uv_v = q[1];
    TexResult r; r.need_perlin = false; r.perlin_idx = 0; r.perlin_scale = 0.f; r.rgb = f3(0, 0, 0);
    if (in_range) r = texture_descend(acc, a.scene.images, a.tex, h);
    const bool need = in_range && r.need_perlin;
    float turb = 0.0f;
    if (a.scene.perlin != nullptr && __any_sync(0xffffffffu, need)) turb = coop_turbulence(a.scene.perlin, need, h.p, r.perlin_idx);
    float3 c = r.need_perlin ? marble(r.perlin_scale, h.p, turb) : r.rgb;
    if (in_range) { a.out[i * 3 + 0] = c.x; a.out[i * 3 + 1] = c.y; a.out[i * 3 + 2] = c.z; }
}

__global__ void rng_kernel(RngKeys keys, uint32_t ka, uint32_t kb, size_t n, float* out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        Rng rng; rng.init(keys, ka, kb);
        for (size_t i = 0; i < n; ++i) out[i] = rng.gen();
    }
}

// FP32 issue ceiling: 8 independent FFMA chains per thread.
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float b, float c) {
    float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            x0 = fmaf(x0, b, c); x1 = fmaf(x1, b, c); x2 = fmaf(x2, b, c); x3 = fmaf(x3, b, c);
            x4 = fmaf(x4, b, c); x5 = fmaf(x5, b, c); x6 = fmaf(x6, b, c); x7 = fmaf(x7, b, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
}


// Read-bandwidth probe: every thread sums float4 loads over a buffer, several passes.  A buffer well inside the 126 MB L2
// measures the L2 ceiling, a much larger one the HBM ceiling (roofline denominators for scenes whose tree lives in global memory).
__global__ void __launch_bounds__(256) read_peak_kernel(const float4* __restrict__ buf, size_t n4, int passes, float* out) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (int p = 0; p < passes; ++p)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
            float4 v = __ldcg(buf + i);                       // .cg: L2 only, so the figure is not an L1 hit rate
            acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
        }
    if (acc.x + acc.y + acc.z + acc.w == 12345.678f) out[0] = acc.x;     // keeps the loads alive
}

}  // namespace b200rt
