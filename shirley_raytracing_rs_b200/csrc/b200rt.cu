// b200rt.cu — the C ABI of include/b200rt.h: scene flattening and upload, BVH build, launch plumbing.
//
// Device code (SURVEY.md §2 "new kernels") lives in the headers this file includes:
//   rt_device.cuh        data layout, math, RNG, intersection, traversal steps, shading, textures
//   render_kernel.cuh    K2 path_trace_kernel_v2   render_scanline + ray_color     (render.rs:17-70)
//   aux_kernels.cuh      K1 closest_hit_kernel     BboxTree::hit_workspace batch   (bvh/bbox_tree.rs:56-91)
//                        K3 resolve_kernel (+ resolve_peers_kernel, flag barrier)  (image.rs:34-40, core/color.rs:31-38)
//                        K4 scatter / camera_rays / texture_value / aabb_hit / rng parity hooks, FFMA-chain microbenchmark
//   lbvh.cuh             K5 linear BVH built on the device                         (bvh/bbox_tree/constructor.rs:9-212)
//   bvh_build.hpp        host binned-SAH builder
//   launch_plan.hpp      CTA size, shared-memory plan, sample-range schedule and grid of a launch (pure host arithmetic)
//   adaptive_plan.hpp    pass schedule and error estimate of tile-adaptive sampling (host and device)
// No tensor cores: nothing on this path is a dense contraction.  No CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "bvh_build.hpp"
#include "launch_plan.hpp"
#include "lbvh.cuh"
#include "rt_device.cuh"

namespace b200rt {

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_last_error = buf;
    return code;
}
#define CU(expr)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (expr);                                                                     \
        if (e_ != cudaSuccess) return fail(e_ == cudaErrorMemoryAllocation ? B200RT_ENOMEM : B200RT_ECUDA, \
                                           "%s: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

}  // namespace b200rt

#include "render_kernel.cuh"
#include "aux_kernels.cuh"


// ==========================================================================================
// host side of the C ABI
// ==========================================================================================
using namespace b200rt;

namespace {

struct Scratch {                     // per in-flight render: counters, events, staging
    Counters* d_counters = nullptr;
    Counters* h_counters = nullptr;  // pinned
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaStream_t launch_stream = nullptr; bool launched = false;   // where the render in flight was enqueued (scene_destroy waits for it)
    float4* d_accum = nullptr; size_t accum_bytes = 0;
    uint8_t* d_rgb = nullptr; size_t rgb_bytes = 0;
    long long* d_fix = nullptr; size_t fix_bytes = 0;  // fixed-point sums of a launch whose tiles are split into sample chunks (adaptive: F)
    long long* d_pass = nullptr; size_t pass_bytes = 0;  // adaptive: the fixed-point sums of one pass (P)
    uint32_t* d_tiles = nullptr; size_t tiles_bytes = 0;  // adaptive: two tile lists, keep flags, tile errors, the active count
    uint32_t launches = 0;
};

}  // namespace

// Scratch objects (pinned counters, events, a stream, frame buffers) are pooled per device
// for the life of the process: creating a scene per frame — what render_scene does — must not
// pay cudaMallocHost / cudaStreamCreate / a 15 MB cudaMalloc every time.
namespace {
std::mutex g_scratch_mu;
std::map<int, std::vector<Scratch*>> g_scratch_pool;
// Scene arenas are pooled the same way: render_scene creates and destroys a scene per frame, and cudaFree is a
// device-wide synchronisation (plus ~0.1 ms) that a 25 ms multi-GPU frame should not pay.  A destroyed scene's
// arena waits here (at most ARENA_POOL_MAX per device) and is handed to the next scene that fits it without
// wasting more than half of it.
struct PooledArena { void* ptr; size_t bytes; };
std::map<int, std::vector<PooledArena>> g_arena_pool;
constexpr size_t ARENA_POOL_MAX = 4;
}  // namespace

struct B200rtScene {
    int device = 0;
    int sm_count = 0;
    size_t smem_optin = 0;
    DeviceScene ds{};
    B200rtSceneInfo info{};
    void* arena = nullptr;        // the one device allocation that holds every scene array
    size_t arena_bytes = 0;       // its capacity (may exceed what this scene uses: pooled arenas are reused)
    std::mutex mu;
    std::map<void*, Scratch*> inflight;   // keyed by stream
    float box_pad = 0.f;          // how far every BVH box was grown
    float max_abs_coord = 0.f;    // largest |coordinate| of any primitive box
};

namespace {

struct DeviceGuard {
    int prev = -1; bool ok = false;
    explicit DeviceGuard(int dev) { if (cudaGetDevice(&prev) == cudaSuccess && cudaSetDevice(dev) == cudaSuccess) ok = true; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

struct DevBuf {   // RAII device buffer for one call
    void* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    int alloc(size_t bytes) { CU(cudaMalloc(&p, bytes ? bytes : 16)); return B200RT_OK; }
    template <class T> T* as() { return reinterpret_cast<T*>(p); }
};

// Buffers kept across calls only grow: when `cap` bytes are too few the old buffer is freed and `bytes` allocated
// (on failure p is null and cap 0).
template <class T> cudaError_t grow(T*& p, size_t& cap, size_t bytes) {
    if (cap >= bytes) return cudaSuccess;
    cudaFree(p); p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
}

// an integer knob from the environment (README.md lists them); unset or empty: the default, the measured best
int env_int(const char* name, int dflt) { const char* v = getenv(name); return v && *v ? atoi(v) : dflt; }

SceneSize scene_size(const B200rtScene* sc) { return {sc->ds.n_nodes, sc->ds.n_prims, sc->ds.n_tex, sc->ds.bvh_depth}; }

// The centre-form (one-FMA) slab planes are conservative only while |origin| * eps stays below the box padding;
// `max_origin` is the largest |coordinate| of a ray origin.  B200RT_FAST_SLAB=0 forces the exact Aabb::hit2 arithmetic.
bool use_fast_slab(const B200rtScene* sc, float max_origin) {
    return sc->box_pad >= 4.0f * 1.1920929e-7f * std::max(sc->max_abs_coord, max_origin) && env_int("B200RT_FAST_SLAB", 1) != 0;
}

int resolve_device(int device, int* out) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(B200RT_ECUDA, "no CUDA device available (%s); this backend has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0) { CU(cudaGetDevice(&device)); }
    if (device >= n) return fail(B200RT_EINVAL, "device %d out of range (%d visible)", device, n);
    *out = device;
    return B200RT_OK;
}

// Layout of the one device allocation that holds every scene array.  Only offsets are assigned here;
// each array is copied straight from where it lies on the host (a host-side staging copy of a
// 1e6-sphere scene — 208 MB, grown piecewise — took 230 ms of scene_create's 360).
struct Arena {
    struct Seg { const void* src; size_t bytes, off; };
    std::vector<Seg> segs;
    size_t total = 0;
    size_t reserve(size_t bytes) { size_t off = (total + 255) & ~size_t(255); total = off + std::max<size_t>(bytes, 16); return off; }
    size_t put(const void* src, size_t bytes) { size_t off = reserve(bytes); if (bytes) segs.push_back({src, bytes, off}); return off; }
    template <class T> size_t put(const std::vector<T>& v) { return put(v.data(), v.size() * sizeof(T)); }   // v must outlive upload()
    cudaError_t upload(uint8_t* dbase) const {
        for (const Seg& g : segs) { cudaError_t e = cudaMemcpy(dbase + g.off, g.src, g.bytes, cudaMemcpyHostToDevice); if (e != cudaSuccess) return e; }
        return cudaSuccess;
    }
};

int validate(const B200rtSceneDesc* d) {
    if (!d) return fail(B200RT_EINVAL, "scene description is NULL");
    if (d->abi_version != B200RT_ABI_VERSION) return fail(B200RT_EINVAL, "abi_version %u != %u", d->abi_version, B200RT_ABI_VERSION);
    if (d->n_prims > B200RT_CODE_ID_MASK) return fail(B200RT_EINVAL, "too many primitives (%u)", d->n_prims);
    if (d->n_prims && (!d->prims || !d->materials)) return fail(B200RT_EINVAL, "prims/materials NULL");
    if ((d->n_spheres && !d->spheres) || (d->n_rects && !d->rects) || (d->n_boxes && !d->boxes) || (d->n_textures && !d->textures) ||
        (d->n_images && !d->images) || (d->n_perlin && !d->perlin))
        return fail(B200RT_EINVAL, "array pointer NULL with non-zero count");
    for (uint32_t i = 0; i < d->n_prims; ++i) {
        const B200rtPrimRef& p = d->prims[i];
        uint32_t lim = p.type == B200RT_PRIM_SPHERE ? d->n_spheres : (p.type == B200RT_PRIM_BOX ? d->n_boxes : (p.type <= B200RT_PRIM_RECT_XZ ? d->n_rects : 0));
        if (p.type > B200RT_PRIM_BOX || p.index >= lim) return fail(B200RT_EINVAL, "prim %u: bad type/index (%u, %u)", i, p.type, p.index);
        if (p.type >= B200RT_PRIM_RECT_XY && p.type <= B200RT_PRIM_RECT_XZ && d->rects[p.index].kind != p.type)
            return fail(B200RT_EINVAL, "prim %u: rect kind %u does not match prim type %u", i, d->rects[p.index].kind, p.type);
        const B200rtMaterial& m = d->materials[i];
        if (m.kind > B200RT_MAT_FAIRY_LIGHT) return fail(B200RT_EINVAL, "prim %u: bad material kind %u", i, m.kind);
        bool textured = m.kind == B200RT_MAT_LAMBERTIAN || m.kind == B200RT_MAT_DIFFUSE_LIGHT || m.kind == B200RT_MAT_FAIRY_LIGHT;
        if (textured && (m.texture < 0 || (uint32_t)m.texture >= d->n_textures)) return fail(B200RT_EINVAL, "prim %u: texture index %d out of range", i, m.texture);
    }
    for (uint32_t t = 0; t < d->n_textures; ++t) {
        const B200rtTexture& x = d->textures[t];
        if (x.kind > B200RT_TEX_CHECKER) return fail(B200RT_EINVAL, "texture %u: bad kind %u", t, x.kind);
        if (x.kind == B200RT_TEX_CHECKER && (x.odd < 0 || x.even < 0 || (uint32_t)x.odd >= t || (uint32_t)x.even >= t))
            return fail(B200RT_EINVAL, "texture %u: checker children must reference lower indices", t);
        if (x.kind == B200RT_TEX_IMAGE && (x.image < 0 || (uint32_t)x.image >= d->n_images)) return fail(B200RT_EINVAL, "texture %u: image index out of range", t);
        if (x.kind == B200RT_TEX_PERLIN && (x.image < 0 || (uint32_t)x.image >= d->n_perlin)) return fail(B200RT_EINVAL, "texture %u: perlin index out of range", t);
    }
    for (uint32_t i = 0; i < d->n_images; ++i)
        if (!d->images[i].rgb8 || d->images[i].width == 0 || d->images[i].height == 0) return fail(B200RT_EINVAL, "image %u: empty", i);
    if (d->skybox.kind > B200RT_SKY_NONE) return fail(B200RT_EINVAL, "bad skybox kind %u", d->skybox.kind);
    return B200RT_OK;
}

DeviceCamera make_camera(const B200rtCamera& c) {
    // camera/mod.rs:98-114 in f64, reduced to the constants the kernel needs
    auto scale3 = [](const double* v, double s, double* o) { o[0] = v[0] * s; o[1] = v[1] * s; o[2] = v[2] * s; };
    double horizontal[3], vertical[3], wf[3], ll[3];
    scale3(c.u, c.width * c.focus_length, horizontal);
    scale3(c.v, c.height * c.focus_length, vertical);
    scale3(c.w, c.focal_length * c.focus_length, wf);
    for (int k = 0; k < 3; ++k) ll[k] = c.origin[k] - horizontal[k] * 0.5 - vertical[k] * 0.5 - wf[k];
    DeviceCamera d;
    auto to3 = [](double x, double y, double z) { return make_float3((float)x, (float)y, (float)z); };
    d.origin = to3(c.origin[0], c.origin[1], c.origin[2]);
    d.llo = to3(ll[0] - c.origin[0], ll[1] - c.origin[1], ll[2] - c.origin[2]);
    double W = (double)c.image_width, H = (double)c.image_height;
    d.hw = to3(horizontal[0] / W, horizontal[1] / W, horizontal[2] / W);
    d.vh = to3(vertical[0] / H, vertical[1] / H, vertical[2] / H);
    double lr = c.lens_radius >= 0 ? c.lens_radius : 0.0;
    d.ul = to3(c.u[0] * lr, c.u[1] * lr, c.u[2] * lr);
    d.vl = to3(c.v[0] * lr, c.v[1] * lr, c.v[2] * lr);
    d.width = c.image_width; d.height = c.image_height;
    d.has_lens = c.lens_radius >= 0 ? 1 : 0;
    return d;
}

int get_scratch(B200rtScene* sc, void* stream_key, Scratch** out) {
    std::lock_guard<std::mutex> lk(sc->mu);
    if (sc->inflight.count(stream_key)) return fail(B200RT_EINVAL, "a render is already in flight on this stream; call b200rt_render_device_finish first");
    Scratch* s = nullptr;
    {
        std::lock_guard<std::mutex> gl(g_scratch_mu);
        auto& pool = g_scratch_pool[sc->device];
        if (!pool.empty()) { s = pool.back(); pool.pop_back(); }
    }
    if (!s) {
        s = new Scratch();
        cudaError_t e = cudaMalloc(&s->d_counters, sizeof(Counters));
        if (e == cudaSuccess) e = cudaMallocHost(&s->h_counters, sizeof(Counters));
        if (e == cudaSuccess) e = cudaEventCreate(&s->ev0);
        if (e == cudaSuccess) e = cudaEventCreate(&s->ev1);
        if (e == cudaSuccess) e = cudaEventCreate(&s->ev2);
        if (e == cudaSuccess) e = cudaEventCreate(&s->ev3);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) { delete s; return fail(B200RT_ECUDA, "scratch allocation: %s", cudaGetErrorString(e)); }
    }
    sc->inflight[stream_key] = s;
    *out = s;
    return B200RT_OK;
}
void put_scratch(B200rtScene* sc, void* stream_key) {
    std::lock_guard<std::mutex> lk(sc->mu);
    auto it = sc->inflight.find(stream_key);
    if (it == sc->inflight.end()) return;
    { std::lock_guard<std::mutex> gl(g_scratch_mu); g_scratch_pool[sc->device].push_back(it->second); }
    sc->inflight.erase(it);
}

// The attribute belongs to the kernel function, not to a launch: host threads rendering different scenes at once would
// lower it under each other's feet if it were set to each launch's own size ("too many resources requested for launch",
// found by tests/test_gpu_scale.py::test_concurrent_renders_from_host_threads).  It is therefore always raised to the device's
// opt-in maximum — the same value from every thread; the carve-out still follows the bytes each launch asks for.
template <class K> int set_smem(K kernel, const B200rtScene* sc, uint32_t bytes) {
    if (bytes > sc->smem_optin) return fail(B200RT_ECUDA, "kernel needs %u B of shared memory, the device offers %zu", bytes, (size_t)sc->smem_optin);
    CU(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sc->smem_optin));
    return B200RT_OK;
}

// The shipped instantiations: {fast, fast + counters, exact + counters} per accessor (and CTA size).  The exact-slab fallback
// always counts: it is the rare path and one variant fewer to compile.  A combination without a kernel is an error.
using RenderKernel = void (*)(RenderArgs);
using HitKernel = void (*)(HitArgs);
template <class Acc, int BLK> RenderKernel render_variant(bool fast, bool count) {
    return !fast ? path_trace_kernel_v2<Acc, true, false, BLK> : count ? path_trace_kernel_v2<Acc, true, true, BLK> : path_trace_kernel_v2<Acc, false, true, BLK>;
}
RenderKernel render_kernel(bool all_in_smem, uint32_t block_threads, bool fast, bool count) {
    if (all_in_smem) return block_threads == 768 ? render_variant<SmemAcc, 768>(fast, count) : nullptr;
    switch (block_threads) {
        case 256: return render_variant<GmemAcc, 256>(fast, count);
        case 512: return render_variant<GmemAcc, 512>(fast, count);
        case 768: return render_variant<GmemAcc, 768>(fast, count);
        default: return nullptr;
    }
}
template <class Acc> HitKernel hit_variant(bool fast, bool count) {
    return !fast ? closest_hit_kernel<Acc, true, false> : count ? closest_hit_kernel<Acc, true, true> : closest_hit_kernel<Acc, false, true>;
}
HitKernel hit_kernel(bool all_in_smem, bool fast, bool count) { return all_in_smem ? hit_variant<SmemAcc>(fast, count) : hit_variant<GmemAcc>(fast, count); }

// One pass of b200rt_render_adaptive: the tiles it renders (NULL: all of them), the fixed-point buffer its sums are added to,
// and the sample count acc_add's clamp is taken for (max_samples, so that the sums of all passes cannot wrap).
struct AdaptivePass { const uint32_t* tile_list; uint32_t n_tiles; long long* fix; uint32_t lim_samples; };

int launch_render(B200rtScene* sc, const B200rtCamera* cam, const B200rtRenderParams* prm, float* d_accum, cudaStream_t stream, Scratch* scr,
                  const AdaptivePass* pass = nullptr) {
    if (cam->image_width == 0 || cam->image_height == 0) return fail(B200RT_EINVAL, "camera image dimensions are zero");
    if ((uint64_t)cam->image_width * cam->image_height > 0xFFFFFFFFull) return fail(B200RT_EINVAL, "image too large");
    RenderArgs a{};
    a.scene = sc->ds;
    a.cam = make_camera(*cam);
    a.keys = rng_keys(prm->seed);
    a.samples = prm->samples == 0 ? 1 : prm->samples;   // src/main.rs:75-80
    a.lim_samples = pass ? pass->lim_samples : a.samples;
    a.tile_list = pass ? pass->tile_list : nullptr;
    a.sample_offset = prm->sample_offset;
    a.max_depth = prm->max_depth;
    uint32_t H = cam->image_height, W = cam->image_width;
    a.row_begin = prm->row_begin; a.row_end = prm->row_end;
    if (a.row_begin == 0 && a.row_end == 0) a.row_end = H;
    if (a.row_end > H || a.row_begin > a.row_end) return fail(B200RT_EINVAL, "row range [%u,%u) outside image height %u", a.row_begin, a.row_end, H);
    a.tiles_x = (W + TILE_W - 1) / TILE_W;
    a.tile_row0 = a.row_begin / TILE_H;
    uint32_t tile_row1 = (a.row_end + TILE_H - 1) / TILE_H;
    a.n_tiles = a.tiles_x * (tile_row1 - a.tile_row0);
    a.shard_count = prm->shard_count == 0 ? 1 : prm->shard_count;
    a.shard_index = prm->shard_index;
    if (a.shard_index >= a.shard_count) return fail(B200RT_EINVAL, "shard_index %u >= shard_count %u", a.shard_index, a.shard_count);
    a.accumulate = (prm->flags & B200RT_FLAG_ACCUMULATE) ? 1 : 0;
    a.accum = reinterpret_cast<float4*>(d_accum);
    a.counters = scr->d_counters;
    bool count = (prm->flags & B200RT_FLAG_COUNT_TRAVERSAL) != 0;
    a.trav_threshold = (uint32_t)std::min(32, std::max(1, env_int("B200RT_TRAV_THRESHOLD", 8)));
    // New paths are handed out only when >= 6 lanes are free (the hand-out block then runs at >= 6 lanes instead of ~5 every
    // iteration): 14.66 -> 15.0 Grays/s on the bench frame, +5 % on the earth frame, 4..8 within 0.5 % of each other.
    a.regen_min = (uint32_t)std::min(32, std::max(1, env_int("B200RT_REGEN_MIN", 6)));
    const bool fast = use_fast_slab(sc, std::max(std::fabs((float)cam->origin[0]), std::max(std::fabs((float)cam->origin[1]), std::fabs((float)cam->origin[2]))));
    const auto [block_threads, plan] = render_shape(scene_size(sc), sc->smem_optin);
    a.plan = plan;
    RenderKernel kernel = render_kernel(plan.all_in_smem, block_threads, fast, count);
    if (!kernel) return fail(B200RT_ECUDA, "no path-tracing kernel is built for %u-thread CTAs with the scene %s", block_threads, plan.all_in_smem ? "in shared memory" : "read through L1");

    scr->launches = 0;
    scr->launch_stream = stream; scr->launched = true;
    CU(cudaEventRecord(scr->ev0, stream));
    CU(cudaMemsetAsync(scr->d_counters, 0, sizeof(Counters), stream));
    // The kernel stores every pixel of the tiles it renders; the buffer is cleared only when some pixels are outside them
    // ("pixels outside the selected rows/tiles are written as zeros", include/b200rt.h).
    const bool covers_frame = a.shard_count == 1 && a.row_begin == 0 && a.row_end == H;
    // (adaptive passes write only through the merge kernel; b200rt_render_adaptive clears the buffer once)
    if (!pass && !a.accumulate && !covers_frame) CU(cudaMemsetAsync(d_accum, 0, (size_t)W * H * sizeof(float4), stream));
    int rc = set_smem(kernel, sc, plan.bytes); if (rc) return rc;
    int blocks_per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, kernel, block_threads, plan.bytes));
    if (blocks_per_sm < 1) return fail(B200RT_ECUDA, "path-tracing kernel does not fit on an SM (smem %u B, %u threads)", plan.bytes, block_threads);
    const uint32_t warps_per_block = block_threads / 32;
    const uint32_t my_tiles = pass ? pass->n_tiles
                            : a.n_tiles > a.shard_index ? (a.n_tiles - a.shard_index + a.shard_count - 1) / a.shard_count : 0u;   // tiles t with t % shard_count == shard_index
    const uint32_t full_grid = (uint32_t)(sc->sm_count * blocks_per_sm);
    const SampleSchedule sched = sample_schedule(a.samples, my_tiles, full_grid * warps_per_block, plan.all_in_smem, env_int("B200RT_CHUNKS", 0));
    a.chunks = sched.chunks;
    a.my_tiles = my_tiles ? my_tiles : 1u;
    std::copy(sched.chunk_begin, sched.chunk_begin + MAX_CHUNKS + 1, a.chunk_begin);
    a.fix = pass ? pass->fix : nullptr;
    if (!pass && a.chunks > 1u) {
        const size_t px = (size_t)W * H;
        cudaError_t e = grow(scr->d_fix, scr->fix_bytes, px * 3 * sizeof(long long));
        if (e != cudaSuccess) return fail(B200RT_ENOMEM, "fixed-point accumulation buffer (%zu px): %s", px, cudaGetErrorString(e));
        a.fix = scr->d_fix;
        CU(cudaMemsetAsync(scr->d_fix, 0, px * 3 * sizeof(long long), stream));
    }
    CU(cudaEventRecord(scr->ev1, stream));
    kernel<<<render_grid(full_grid, my_tiles, a.chunks, warps_per_block), block_threads, plan.bytes, stream>>>(a);
    CU(cudaGetLastError());
    scr->launches += 1;
    if (!pass && a.chunks > 1u && a.row_end > a.row_begin) {
        dim3 fb(128, 1), fg((W + 127) / 128, a.row_end - a.row_begin);
        finalize_kernel<<<fg, fb, 0, stream>>>(a);
        CU(cudaGetLastError());
        scr->launches += 1;
    }
    CU(cudaEventRecord(scr->ev2, stream));
    CU(cudaMemcpyAsync(scr->h_counters, scr->d_counters, sizeof(Counters), cudaMemcpyDeviceToHost, stream));
    return B200RT_OK;
}

int finish_render(Scratch* scr, cudaStream_t stream, cudaEvent_t end_event, B200rtStats* stats) {
    CU(cudaStreamSynchronize(stream));
    scr->launched = false;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->rays = scr->h_counters->rays; stats->paths = scr->h_counters->paths;
        stats->node_visits = scr->h_counters->nodes; stats->prim_tests = scr->h_counters->prims;
        stats->depth_exhausted = scr->h_counters->exhausted;
        for (int k = 0; k < 8; ++k) stats->diag[k] = scr->h_counters->diag[k];
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, scr->ev1, scr->ev2)); stats->kernel_ms = ms;
        CU(cudaEventElapsedTime(&ms, scr->ev0, end_event)); stats->total_ms = ms;
        stats->launches = scr->launches;
    }
    return B200RT_OK;
}

}  // namespace

extern "C" {

int b200rt_resolve_rgb8_device(const float* d_accum, uint32_t W, uint32_t H, uint32_t samples, uint8_t* d_out, void* cuda_stream);
int b200rt_resolve_peers_rgb8_device(const float* const* d_accums, uint32_t n_peers, uint32_t W, uint32_t H, uint32_t samples,
                                     uint32_t row_begin, uint32_t row_end, uint8_t* d_out, const uint32_t* d_my_flags, void* cuda_stream);

const char* b200rt_last_error(void) { return g_last_error.c_str(); }
int b200rt_abi_version(void) { return B200RT_ABI_VERSION; }
int b200rt_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int b200rt_scene_create(const B200rtSceneDesc* d, int device, B200rtScene** out) {
    if (!out) return fail(B200RT_EINVAL, "out is NULL");
    *out = nullptr;
    // B200RT_TIMING=1: wall time of each phase on stderr (large scenes: where scene_create's time goes)
    const bool timing = getenv("B200RT_TIMING") != nullptr;
    auto t_prev = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[b200rt] scene_create %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t_prev).count());
        t_prev = now;
    };
    int rc = validate(d); if (rc) return rc;
    lap("validate");
    rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    if (!guard.ok) return fail(B200RT_ECUDA, "cudaSetDevice(%d) failed", device);

    std::vector<GeomRec> geom(d->n_prims);
    std::vector<MatRec> mats(d->n_prims);
    std::vector<BuildPrim> bprims;
    std::vector<BuildPrim> bp_all(d->n_prims);       // one slot per primitive (code < 0: no leaf), compacted below
    float max_abs = 0.f;
#pragma omp parallel for schedule(static) reduction(max : max_abs) if (d->n_prims >= 65536)
    for (long long ii = 0; ii < (long long)d->n_prims; ++ii) {
        const uint32_t i = (uint32_t)ii;
        const B200rtPrimRef& p = d->prims[i];
        GeomRec g{}; HostBox b{};
        if (p.type == B200RT_PRIM_SPHERE) {
            const B200rtSphere& s = d->spheres[p.index];
            g.g0 = make_float4(s.cx, s.cy, s.cz, s.radius);
            // sphere.rs:54-60: center -/+ (r,r,r); a negative radius yields an inverted box
            b.lo[0] = s.cx - s.radius; b.lo[1] = s.cy - s.radius; b.lo[2] = s.cz - s.radius;
            b.hi[0] = s.cx + s.radius; b.hi[1] = s.cy + s.radius; b.hi[2] = s.cz + s.radius;
        } else if (p.type == B200RT_PRIM_BOX) {
            const B200rtBox& x = d->boxes[p.index];
            g.g0 = make_float4(x.min[0], x.min[1], x.min[2], 0.f);
            g.g1 = make_float4(x.max[0], x.max[1], x.max[2], 0.f);
            for (int k = 0; k < 3; ++k) { b.lo[k] = x.min[k]; b.hi[k] = x.max[k]; }   // rect.rs:158-163
        } else {
            const B200rtRect& r = d->rects[p.index];
            g.g0 = make_float4(r.d1_min, r.d1_max, r.d2_min, r.d2_max);
            g.g1 = make_float4(r.offset, 0.f, 0.f, 0.f);
            int d1 = p.type == B200RT_PRIM_RECT_YZ ? 1 : 0, d2 = p.type == B200RT_PRIM_RECT_XY ? 1 : 2, dn = 3 - d1 - d2;
            b.lo[d1] = r.d1_min; b.hi[d1] = r.d1_max; b.lo[d2] = r.d2_min; b.hi[d2] = r.d2_max;
            b.lo[dn] = r.offset - 0.0001f; b.hi[dn] = r.offset + 0.0001f;             // rect.rs:9,82-99
        }
        geom[i] = g;
        const B200rtMaterial& m = d->materials[i];
        MatRec mr{};
        mr.kind = m.kind; mr.tex = -1;
        mr.m0 = make_float4(m.albedo[0], m.albedo[1], m.albedo[2], m.param);
        if (m.kind == B200RT_MAT_METAL) mr.m0.w = m.param > 1.0f ? 1.0f : m.param;   // metal.rs:18-21
        if (m.kind == B200RT_MAT_LAMBERTIAN || m.kind == B200RT_MAT_DIFFUSE_LIGHT || m.kind == B200RT_MAT_FAIRY_LIGHT) {
            const B200rtTexture& t = d->textures[m.texture];
            if (t.kind == B200RT_TEX_SOLID) mr.m0 = make_float4(t.rgb[0], t.rgb[1], t.rgb[2], 0.f);   // resolved at upload
            else mr.tex = m.texture;
        }
        mats[i] = mr;
        // the reference keeps inverted boxes in its tree, where Aabb::hit2 can never pass;
        // here they simply get no leaf.  NaN boxes likewise.
        bool valid = true;
        for (int k = 0; k < 3; ++k) valid = valid && (b.lo[k] <= b.hi[k]);
        BuildPrim bp; bp.box = b; bp.code = valid ? (int)((p.type << B200RT_LEAF_TYPE_SHIFT) | i) : -1;
        for (int k = 0; k < 3; ++k) { bp.centroid[k] = 0.5f * (b.lo[k] + b.hi[k]); if (valid) max_abs = std::max(max_abs, std::max(std::fabs(b.lo[k]), std::fabs(b.hi[k]))); }
        bp_all[i] = bp;
    }
    bprims.reserve(d->n_prims);
    for (const BuildPrim& bp : bp_all) if (bp.code >= 0) bprims.push_back(bp);
    std::vector<BuildPrim>().swap(bp_all);
    lap("flatten prims + materials");
    // Scene-spanning primitives leave the BVH for the up-front list (DeviceScene::top_prims):
    // a box whose surface area is >= 30 % of the whole scene's is met by nearly every ray.
    DeviceScene ds_top{};
    {
        HostBox all; detail::box_init(all);
        for (auto& bp : bprims) detail::box_grow(all, bp.box);
        float total = detail::box_area(all);
        std::vector<BuildPrim> kept;
        kept.reserve(bprims.size());
        for (auto& bp : bprims) {
            if (bprims.size() > 2 && ds_top.n_top_prims < 7 && total > 0.f && detail::box_area(bp.box) >= 0.3f * total)
                ds_top.top_prims[ds_top.n_top_prims++] = ~bp.code;
            else kept.push_back(bp);
        }
        bprims.swap(kept);
    }
    // Grow boxes by 4e-6 x the scene's largest coordinate (~34 ulp): the f32 slab tests are
    // then conservative with respect to the f32 primitive tests — for the exact form always,
    // for the one-FMA form (extra error eps * |origin| per axis) while ray origins stay
    // within ~8x the scene extent (checked per launch).  A box only culls.
    float pad = max_abs * 4e-6f;
    for (auto& bp : bprims) for (int k = 0; k < 3; ++k) { bp.box.lo[k] -= pad; bp.box.hi[k] += pad; }
    // Builder: binned SAH on the host (bvh_build.hpp), or — for scenes large enough that the host build
    // would dominate a frame — the linear BVH built on the device (lbvh.cuh).  B200RT_BUILDER=sah|lbvh forces one.
    bool use_lbvh = bprims.size() >= LBVH_AUTO_MIN;
    if (const char* v = getenv("B200RT_BUILDER")) { if (!strcmp(v, "lbvh")) use_lbvh = true; else if (!strcmp(v, "sah")) use_lbvh = false; }
    if (bprims.size() < 2) use_lbvh = false;
    HostBox lbvh_bounds; detail::box_init(lbvh_bounds);
    std::vector<BuildPrim> lbvh_prims;
    BvhBuildResult bvh;
    float host_build_ms = 0.f;
    if (use_lbvh) {
        for (auto& bp : bprims) detail::box_grow(lbvh_bounds, bp.box);
        lbvh_prims.swap(bprims);
    } else {
        auto t0 = std::chrono::steady_clock::now();
        bvh = build_bvh(std::move(bprims));
        host_build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (bvh.depth > BVH_MAX_DEPTH) return fail(B200RT_ESTACK, "BVH depth %u exceeds the traversal stack", bvh.depth);
    }

    lap(use_lbvh ? "top list + padding" : "top list + padding + host SAH");
    std::vector<TexRec> tex(d->n_textures);
    for (uint32_t t = 0; t < d->n_textures; ++t) {
        const B200rtTexture& x = d->textures[t];
        TexRec r{}; r.kind = x.kind; r.r = x.rgb[0]; r.g = x.rgb[1]; r.b = x.rgb[2]; r.scalar = x.scalar; r.odd = x.odd; r.even = x.even; r.image = x.image;
        tex[t] = r;
    }

    B200rtScene* sc = new B200rtScene();
    sc->device = device;
    auto bail = [&](int code) { b200rt_scene_destroy(sc); return code; };
    {   // cudaGetDeviceProperties costs 3-160 ms per call on this driver: two attribute queries instead
        int sms = 0, optin = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess ||
            cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device) != cudaSuccess)
            return bail(fail(B200RT_ECUDA, "cudaDeviceGetAttribute failed"));
        sc->sm_count = sms; sc->smem_optin = (size_t)optin;
    }

    static_assert(sizeof(HostNode) == sizeof(BvhNode), "node layout");
    // The device's copy of the tree: each child box as centre + half-extent (rt_device.cuh: aabb_center),
    // re-derived outwards from the builder's (lo, hi): c = (lo+hi)/2, h = max(hi - c, c - lo) bumped up one ulp,
    // so [c - h, c + h] contains [lo, hi].  An empty child (lo > hi) gets h = -1: near > far on every axis, never
    // entered.  ONE copy is uploaded; the exact-slab fallback derives (c - h, c + h) on the fly.
    auto centre_form = [](const std::vector<HostNode>& src) {
        std::vector<BvhNode> out(src.size());
#pragma omp parallel for schedule(static) if (src.size() >= 65536)
        for (long long i = 0; i < (long long)src.size(); ++i) {
            const float* q = reinterpret_cast<const float*>(&src[i]);
            float* o = reinterpret_cast<float*>(&out[i]);
            for (int ch = 0; ch < 2; ++ch) {
                const float* lo = q + 6 * ch; const float* hi = lo + 3;
                for (int k = 0; k < 3; ++k) {
                    float c = 0.f, h = -1.f;
                    if (lo[k] <= hi[k]) {
                        c = 0.5f * lo[k] + 0.5f * hi[k];
                        h = std::nextafterf(std::max(hi[k] - c, c - lo[k]), INFINITY);
                        if (!std::isfinite(c) || !std::isfinite(h)) { c = 0.f; h = 3.0e38f; }   // unbounded box: always entered
                    }
                    o[6 * ch + k] = c; o[6 * ch + 3 + k] = h;
                }
            }
            o[12] = q[12]; o[13] = q[13]; o[14] = q[14]; o[15] = q[15];
        }
        return out;
    };
    const size_t n_nodes = use_lbvh ? lbvh_prims.size() - 1 : bvh.nodes.size();
    std::vector<BvhNode> cnodes;
    if (!use_lbvh) cnodes = centre_form(bvh.nodes);
    lap("centre/half-extent nodes");
    Arena arena;
    size_t off_nodes = use_lbvh ? arena.reserve(n_nodes * sizeof(BvhNode)) : arena.put(cnodes);
    size_t off_geom = arena.put(geom), off_mats = arena.put(mats), off_tex = arena.put(tex);
    // images: RGB8 -> RGBA8 so a texel is one 4-byte load
    std::vector<ImageRec> images(d->n_images);
    std::vector<size_t> off_img(d->n_images);
    std::vector<std::vector<uchar4>> rgba(d->n_images);
    for (uint32_t i = 0; i < d->n_images; ++i) {
        const B200rtImage& im = d->images[i];
        size_t n = (size_t)im.width * im.height;
        rgba[i].resize(n);
        for (size_t k = 0; k < n; ++k) rgba[i][k] = make_uchar4(im.rgb8[3 * k], im.rgb8[3 * k + 1], im.rgb8[3 * k + 2], 255);
        off_img[i] = arena.put(rgba[i]);
        images[i].width = im.width; images[i].height = im.height; images[i].pad = 0;
    }
    std::vector<PerlinRec> perlin(d->n_perlin);
    for (uint32_t i = 0; i < d->n_perlin; ++i) {
        for (int k = 0; k < 256; ++k) perlin[i].ranfloat[k] = make_float4(d->perlin[i].ranfloat[k][0], d->perlin[i].ranfloat[k][1], d->perlin[i].ranfloat[k][2], 0.f);
        memcpy(perlin[i].perm_x, d->perlin[i].perm_x, 256); memcpy(perlin[i].perm_y, d->perlin[i].perm_y, 256); memcpy(perlin[i].perm_z, d->perlin[i].perm_z, 256);
    }
    size_t off_perlin = arena.put(perlin);
    size_t off_images = arena.put(images);      // the texel pointers are filled in below, before the upload
    lap("lay out arena");
    uint8_t* dbase = nullptr;
    {
        size_t capacity = 0;
        {   // a pooled arena of a destroyed scene, if one fits
            std::lock_guard<std::mutex> gl(g_scratch_mu);
            auto& pool = g_arena_pool[device];
            for (size_t k = 0; k < pool.size(); ++k)
                if (pool[k].bytes >= arena.total && pool[k].bytes <= 2 * arena.total + (1u << 20)) {
                    dbase = static_cast<uint8_t*>(pool[k].ptr); capacity = pool[k].bytes;
                    pool.erase(pool.begin() + k);
                    break;
                }
        }
        cudaError_t e = cudaSuccess;
        if (!dbase) { e = cudaMalloc(&dbase, arena.total); capacity = arena.total; }
        if (e != cudaSuccess) return bail(fail(B200RT_ENOMEM, "scene arena (%zu B): %s", arena.total, cudaGetErrorString(e)));
        sc->arena = dbase; sc->arena_bytes = capacity;
        for (uint32_t i = 0; i < d->n_images; ++i) images[i].texels = reinterpret_cast<const uchar4*>(dbase + off_img[i]);
        e = arena.upload(dbase);
        if (e != cudaSuccess) return bail(fail(B200RT_ECUDA, "scene upload: %s", cudaGetErrorString(e)));
        sc->info.device_bytes = arena.total;
    }
    lap("cudaMalloc + H2D");
    sc->ds.nodes = reinterpret_cast<const BvhNode*>(dbase + off_nodes);
    if (use_lbvh) {
        uint32_t depth = 0; float ms = 0.f;
        cudaError_t e = lbvh::build(lbvh_prims, lbvh_bounds, reinterpret_cast<BvhNode*>(dbase + off_nodes), &depth, &ms);
        if (e != cudaSuccess) return bail(fail(e == cudaErrorMemoryAllocation ? B200RT_ENOMEM : B200RT_ECUDA, "device BVH build: %s", cudaGetErrorString(e)));
        sc->info.bvh_build_ms = ms; sc->info.bvh_builder = 1;
        lap("device LBVH (incl. its uploads)");
        const char* force = getenv("B200RT_LBVH_MAX_DEPTH");      // test hook: pretend the stack is shallower
        const uint32_t limit = force && *force ? (uint32_t)atoi(force) : BVH_MAX_DEPTH;
        if (depth > limit) {
            // A linear BVH over strongly clustered primitives (many equal Morton prefixes) can be deeper than the
            // traversal stack.  The host builder bounds its depth (median splits near the limit): rebuild with it into
            // the same node slots (both builders emit n - 1 nodes) instead of failing.
            auto t0 = std::chrono::steady_clock::now();
            bvh = build_bvh(std::move(lbvh_prims));
            host_build_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
            if (bvh.depth > BVH_MAX_DEPTH || bvh.nodes.size() != n_nodes) return bail(fail(B200RT_ESTACK, "BVH depth %u exceeds the traversal stack", bvh.depth));
            cnodes = centre_form(bvh.nodes);
            e = cudaMemcpy(dbase + off_nodes, cnodes.data(), n_nodes * sizeof(BvhNode), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) return bail(fail(B200RT_ECUDA, "scene upload: %s", cudaGetErrorString(e)));
            sc->info.bvh_build_ms = host_build_ms; sc->info.bvh_builder = 0;
            lap("host SAH rebuild (device tree too deep)");
        } else bvh.depth = depth;
    } else { sc->info.bvh_build_ms = host_build_ms; sc->info.bvh_builder = 0; }
    sc->ds.geom = reinterpret_cast<const GeomRec*>(dbase + off_geom);
    sc->ds.mats = reinterpret_cast<const MatRec*>(dbase + off_mats);
    sc->ds.tex = reinterpret_cast<const TexRec*>(dbase + off_tex);
    sc->ds.images = reinterpret_cast<const ImageRec*>(dbase + off_images);
    sc->ds.perlin = d->n_perlin ? reinterpret_cast<const PerlinRec*>(dbase + off_perlin) : nullptr;
    sc->ds.n_perlin = d->n_perlin;
    sc->ds.n_top_prims = ds_top.n_top_prims;
    for (int k = 0; k < 7; ++k) sc->ds.top_prims[k] = ds_top.top_prims[k];
    sc->box_pad = pad; sc->max_abs_coord = max_abs;
    sc->ds.n_nodes = (uint32_t)n_nodes; sc->ds.n_prims = d->n_prims; sc->ds.n_tex = d->n_textures; sc->ds.bvh_depth = bvh.depth;
    sc->ds.sky_kind = d->skybox.kind == B200RT_SKY_ABOVE ? B200RT_SKY_ABOVE : B200RT_SKY_FLAT;
    sc->ds.has_emitters = 0;      // DiffuseLight / FairyLight present: ray_color's `emitted` accumulator is live (render kernel)
    for (uint32_t i = 0; i < d->n_prims; ++i)
        if (d->materials[i].kind == B200RT_MAT_DIFFUSE_LIGHT || d->materials[i].kind == B200RT_MAT_FAIRY_LIGHT) { sc->ds.has_emitters = 1; break; }
    bool flat = d->skybox.kind == B200RT_SKY_FLAT;
    sc->ds.sky_r = flat ? d->skybox.rgb[0] : 0.f; sc->ds.sky_g = flat ? d->skybox.rgb[1] : 0.f; sc->ds.sky_b = flat ? d->skybox.rgb[2] : 0.f;
    sc->info.n_prims = d->n_prims; sc->info.n_bvh_nodes = sc->ds.n_nodes; sc->info.bvh_depth = bvh.depth;
    sc->info.bvh_nodes_in_smem = hook_plan(scene_size(sc), sc->smem_optin).n_top;
    *out = sc;
    return B200RT_OK;
}

void b200rt_scene_destroy(B200rtScene* sc) {
    if (!sc) return;
    DeviceGuard guard(sc->device);
    {   // renders still in flight on this scene: wait, then return their scratch to the pool
        std::lock_guard<std::mutex> gl(g_scratch_mu);
        for (auto& kv : sc->inflight) {
            // the arena goes back to a pool and may be overwritten by the next scene: nothing may still read it
            if (kv.second->launched) cudaStreamSynchronize(kv.second->launch_stream);
            kv.second->launched = false;
            g_scratch_pool[sc->device].push_back(kv.second);
        }
    }
    if (sc->arena) {   // one arena holds every scene array: back to the pool (every render on it has been waited for above)
        bool pooled = false;
        {
            std::lock_guard<std::mutex> gl(g_scratch_mu);
            auto& pool = g_arena_pool[sc->device];
            if (pool.size() < ARENA_POOL_MAX) { pool.push_back({sc->arena, sc->arena_bytes}); pooled = true; }
        }
        if (!pooled) cudaFree(sc->arena);
    }
    delete sc;
}

int b200rt_scene_info(const B200rtScene* sc, B200rtSceneInfo* out) {
    if (!sc || !out) return fail(B200RT_EINVAL, "NULL argument");
    *out = sc->info;
    return B200RT_OK;
}

int b200rt_render_device(const B200rtScene* csc, const B200rtCamera* cam, const B200rtRenderParams* prm, float* d_accum, void* cuda_stream) {
    if (!csc || !cam || !prm || !d_accum) return fail(B200RT_EINVAL, "NULL argument");
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    DeviceGuard guard(sc->device);
    Scratch* scr; int rc = get_scratch(sc, cuda_stream, &scr); if (rc) return rc;
    rc = launch_render(sc, cam, prm, d_accum, (cudaStream_t)cuda_stream, scr);
    if (rc) put_scratch(sc, cuda_stream);
    return rc;
}

int b200rt_render_device_finish(const B200rtScene* csc, void* cuda_stream, B200rtStats* stats) {
    if (!csc) return fail(B200RT_EINVAL, "NULL argument");
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    DeviceGuard guard(sc->device);
    Scratch* scr = nullptr;
    { std::lock_guard<std::mutex> lk(sc->mu); auto it = sc->inflight.find(cuda_stream); if (it != sc->inflight.end()) scr = it->second; }
    if (!scr) return fail(B200RT_EINVAL, "no render in flight on this stream");
    int rc = finish_render(scr, (cudaStream_t)cuda_stream, scr->ev2, stats);
    put_scratch(sc, cuda_stream);
    return rc;
}

static int render_host_impl(const B200rtScene* csc, const B200rtCamera* cam, const B200rtRenderParams* prm, float* accum, uint8_t* out_rgb8, B200rtStats* stats) {
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    int device = sc->device;
    if (prm->device >= 0 && prm->device != device) return fail(B200RT_EINVAL, "params.device %d != scene device %d", prm->device, device);
    DeviceGuard guard(device);
    int key_local; void* key = &key_local;   // private key: concurrent host threads never collide
    Scratch* scr; int rc = get_scratch(sc, key, &scr); if (rc) return rc;
    size_t px = (size_t)cam->image_width * cam->image_height;
    auto done = [&](int code) { put_scratch(sc, key); return code; };
    if (cudaError_t e = grow(scr->d_accum, scr->accum_bytes, px * sizeof(float4)))
        return done(fail(B200RT_ENOMEM, "accumulation buffer (%zu px): %s", px, cudaGetErrorString(e)));
    if (out_rgb8) {
        if (cudaError_t e = grow(scr->d_rgb, scr->rgb_bytes, px * 3)) return done(fail(B200RT_ENOMEM, "rgb8 buffer: %s", cudaGetErrorString(e)));
    }
    // Progressive rendering with host buffers: with B200RT_FLAG_ACCUMULATE the caller's float4 sums
    // (an earlier call's output, or a checkpoint) are uploaded first and the new samples are added.
    B200rtRenderParams p = *prm;
    const bool progressive = (p.flags & B200RT_FLAG_ACCUMULATE) && accum;
    if (!progressive) p.flags &= ~B200RT_FLAG_ACCUMULATE;
    if (progressive) {
        cudaError_t eu = cudaMemcpyAsync(scr->d_accum, accum, px * sizeof(float4), cudaMemcpyHostToDevice, scr->own_stream);
        if (eu != cudaSuccess) return done(fail(B200RT_ECUDA, "H2D copy of the accumulation buffer: %s", cudaGetErrorString(eu)));
    }
    rc = launch_render(sc, cam, &p, reinterpret_cast<float*>(scr->d_accum), scr->own_stream, scr);
    if (rc) return done(rc);
    cudaError_t e = cudaSuccess;
    if (out_rgb8) {
        // progressive: n = the summed sample count in .w
        rc = b200rt_resolve_rgb8_device(reinterpret_cast<float*>(scr->d_accum), cam->image_width, cam->image_height, progressive ? 0 : (p.samples == 0 ? 1 : p.samples), scr->d_rgb, scr->own_stream);
        if (rc) return done(rc);
        scr->launches += 1;
        e = cudaMemcpyAsync(out_rgb8, scr->d_rgb, px * 3, cudaMemcpyDeviceToHost, scr->own_stream);
    }
    if (e == cudaSuccess && accum) e = cudaMemcpyAsync(accum, scr->d_accum, px * sizeof(float4), cudaMemcpyDeviceToHost, scr->own_stream);
    if (e == cudaSuccess) e = cudaEventRecord(scr->ev3, scr->own_stream);
    if (e != cudaSuccess) return done(fail(B200RT_ECUDA, "D2H copy: %s", cudaGetErrorString(e)));
    rc = finish_render(scr, scr->own_stream, scr->ev3, stats);
    return done(rc);
}

int b200rt_render(const B200rtScene* csc, const B200rtCamera* cam, const B200rtRenderParams* prm, float* accum, B200rtStats* stats) {
    if (!csc || !cam || !prm || !accum) return fail(B200RT_EINVAL, "NULL argument");
    return render_host_impl(csc, cam, prm, accum, nullptr, stats);
}

int b200rt_render_rgb8(const B200rtScene* csc, const B200rtCamera* cam, const B200rtRenderParams* prm, uint8_t* out_rgb8, float* accum, B200rtStats* stats) {
    if (!csc || !cam || !prm || !out_rgb8) return fail(B200RT_EINVAL, "NULL argument");
    return render_host_impl(csc, cam, prm, accum, out_rgb8, stats);
}

// Tile-adaptive sampling (b200rt_render_adaptive): passes over the still-active tiles (adaptive_plan.hpp), each one K2 launch over the tile list, the merge
// kernel (estimate, F += P, stopped tiles' pixels) and the compaction of the next list; the host reads the active count after
// each pass.  Pass 0 adds straight into F and renders every tile; pass 1 still renders every tile, so it needs no list either.
static int render_adaptive_impl(B200rtScene* sc, const B200rtCamera* cam, const B200rtRenderParams* prm, const B200rtAdaptiveParams* ad,
                                float* accum, uint8_t* out_rgb8, float* tile_error, B200rtStats* stats, Scratch* scr) {
    const uint32_t W = cam->image_width, H = cam->image_height;
    uint32_t row_begin = prm->row_begin, row_end = prm->row_end;
    if (row_begin == 0 && row_end == 0) row_end = H;
    const uint32_t tiles_x = (W + TILE_W - 1) / TILE_W, tile_row0 = row_begin / TILE_H, tile_row1 = (row_end + TILE_H - 1) / TILE_H;
    const uint32_t n_tiles = row_end > row_begin ? tiles_x * (tile_row1 - tile_row0) : 0u;
    const size_t px = (size_t)W * H;
    cudaError_t e = grow(scr->d_accum, scr->accum_bytes, px * sizeof(float4));
    if (e == cudaSuccess) e = grow(scr->d_fix, scr->fix_bytes, px * 3 * sizeof(long long));
    if (e == cudaSuccess) e = grow(scr->d_pass, scr->pass_bytes, px * 3 * sizeof(long long));
    if (e == cudaSuccess) e = grow(scr->d_tiles, scr->tiles_bytes, ((size_t)n_tiles * 4 + 1) * sizeof(uint32_t));
    if (e == cudaSuccess && out_rgb8) e = grow(scr->d_rgb, scr->rgb_bytes, px * 3);
    if (e != cudaSuccess) return fail(B200RT_ENOMEM, "adaptive sampling buffers (%zu px): %s", px, cudaGetErrorString(e));
    uint32_t* lists[2] = {scr->d_tiles, scr->d_tiles + n_tiles};
    uint32_t* keep = scr->d_tiles + 2 * (size_t)n_tiles;
    float* d_err = reinterpret_cast<float*>(scr->d_tiles + 3 * (size_t)n_tiles);
    uint32_t* d_count = scr->d_tiles + 4 * (size_t)n_tiles;
    cudaStream_t stream = scr->own_stream;
    // ev3 marks the start of the call; launch_render records ev0..ev2 per pass, and ev0 is recorded again to mark the end
    CU(cudaEventRecord(scr->ev3, stream));
    CU(cudaMemsetAsync(scr->d_accum, 0, px * sizeof(float4), stream));
    CU(cudaMemsetAsync(scr->d_fix, 0, px * 3 * sizeof(long long), stream));
    CU(cudaMemsetAsync(scr->d_pass, 0, px * 3 * sizeof(long long), stream));

    B200rtRenderParams p = *prm;
    p.flags &= B200RT_FLAG_COUNT_TRAVERSAL; p.shard_count = 1; p.shard_index = 0; p.row_begin = row_begin; p.row_end = row_end;
    B200rtStats sum{};
    uint32_t n_prev = 0, active = n_tiles, launches = 0, which = 0;
    const uint32_t* list = nullptr;
    for (uint32_t k = 0; active > 0; ++k) {
        const uint32_t n = adaptive_samples_after(ad->initial_samples, ad->max_samples, k);
        p.samples = n - n_prev; p.sample_offset = prm->sample_offset + n_prev;
        const AdaptivePass pass{list, active, k == 0 ? scr->d_fix : scr->d_pass, ad->max_samples};
        if (int rc = launch_render(sc, cam, &p, reinterpret_cast<float*>(scr->d_accum), stream, scr, &pass)) return rc;
        launches += scr->launches;
        uint32_t next = active;
        if (k > 0) {
            MergeArgs m{};
            m.list = list; m.n_active = active; m.F = scr->d_fix; m.P = scr->d_pass; m.accum = scr->d_accum; m.tile_error = d_err; m.keep = keep;
            m.n = n_prev; m.s = n - n_prev; m.last = n == ad->max_samples ? 1u : 0u; m.threshold = ad->threshold;
            m.W = W; m.row_begin = row_begin; m.row_end = row_end; m.tiles_x = tiles_x; m.tile_row0 = tile_row0;
            adaptive_merge_kernel<<<(active + 7) / 8, 256, 0, stream>>>(m);
            CU(cudaGetLastError());
            adaptive_compact_kernel<<<1, COMPACT_THREADS, 0, stream>>>(list, keep, active, lists[which], d_count);
            CU(cudaGetLastError());
            launches += 2;
            CU(cudaMemcpyAsync(&next, d_count, sizeof next, cudaMemcpyDeviceToHost, stream));
        }
        CU(cudaStreamSynchronize(stream));
        const Counters& c = *scr->h_counters;
        sum.rays += c.rays; sum.paths += c.paths; sum.node_visits += c.nodes; sum.prim_tests += c.prims; sum.depth_exhausted += c.exhausted;
        for (int d = 0; d < 8; ++d) sum.diag[d] += c.diag[d];
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, scr->ev1, scr->ev2)); sum.kernel_ms += ms;
        if (k > 0) { list = lists[which]; which ^= 1u; }
        active = next; n_prev = n;
    }
    if (out_rgb8) {
        if (int rc = b200rt_resolve_rgb8_device(reinterpret_cast<float*>(scr->d_accum), W, H, 0, scr->d_rgb, stream)) return rc;
        launches += 1;
        e = cudaMemcpyAsync(out_rgb8, scr->d_rgb, px * 3, cudaMemcpyDeviceToHost, stream);
    }
    if (e == cudaSuccess && accum) e = cudaMemcpyAsync(accum, scr->d_accum, px * sizeof(float4), cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess && tile_error) {
        // tiles with no selected pixel: -1; the others sit in one contiguous block of tile rows
        std::fill(tile_error, tile_error + (size_t)tiles_x * ((H + TILE_H - 1) / TILE_H), -1.0f);
        if (n_tiles) e = cudaMemcpyAsync(tile_error + (size_t)tile_row0 * tiles_x, d_err, n_tiles * sizeof(float), cudaMemcpyDeviceToHost, stream);
    }
    if (e == cudaSuccess) e = cudaEventRecord(scr->ev0, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) return fail(B200RT_ECUDA, "adaptive sampling copy-back: %s", cudaGetErrorString(e));
    if (stats) {
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, scr->ev3, scr->ev0));
        sum.total_ms = ms;
        sum.launches = launches;
        *stats = sum;
    }
    return B200RT_OK;
}

int b200rt_render_adaptive(const B200rtScene* csc, const B200rtCamera* cam, const B200rtRenderParams* prm, const B200rtAdaptiveParams* ad,
                           float* accum, uint8_t* out_rgb8, float* tile_error, B200rtStats* stats) {
    if (!csc || !cam || !prm || !ad) return fail(B200RT_EINVAL, "NULL argument");
    if (prm->flags & B200RT_FLAG_ACCUMULATE) return fail(B200RT_EINVAL, "adaptive sampling cannot add to an earlier result (B200RT_FLAG_ACCUMULATE)");
    if (prm->shard_count > 1) return fail(B200RT_EINVAL, "adaptive sampling renders whole frames: shard_count %u is not supported", prm->shard_count);
    if (ad->initial_samples == 0) return fail(B200RT_EINVAL, "adaptive initial_samples is 0");
    if (ad->max_samples <= ad->initial_samples) return fail(B200RT_EINVAL, "adaptive max_samples %u must exceed initial_samples %u", ad->max_samples, ad->initial_samples);
    if (!(ad->threshold >= 0.0f) || !std::isfinite(ad->threshold)) return fail(B200RT_EINVAL, "adaptive threshold %g must be finite and >= 0", (double)ad->threshold);
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    if (prm->device >= 0 && prm->device != sc->device) return fail(B200RT_EINVAL, "params.device %d != scene device %d", prm->device, sc->device);
    const uint32_t W = cam->image_width, H = cam->image_height;
    if (W == 0 || H == 0) return fail(B200RT_EINVAL, "camera image dimensions are zero");
    if ((uint64_t)W * H > 0xFFFFFFFFull) return fail(B200RT_EINVAL, "image too large");
    const uint32_t row_end = prm->row_begin == 0 && prm->row_end == 0 ? H : prm->row_end;
    if (row_end > H || prm->row_begin > row_end) return fail(B200RT_EINVAL, "row range [%u,%u) outside image height %u", prm->row_begin, row_end, H);

    DeviceGuard guard(sc->device);
    int key_local; void* key = &key_local;   // private key: concurrent host threads never collide
    Scratch* scr; int rc = get_scratch(sc, key, &scr); if (rc) return rc;
    rc = render_adaptive_impl(sc, cam, prm, ad, accum, out_rgb8, tile_error, stats, scr);
    if (rc) cudaStreamSynchronize(scr->own_stream);   // nothing of a failed call may still run when its scratch is reused
    scr->launched = false;
    put_scratch(sc, key);
    return rc;
}

// ---- render_scene on several GPUs from ONE host process (what a `ray-cli` user has) -------------------------------
// B200rtMulti keeps, for a fixed device list, everything a frame loop would otherwise re-create per call: one worker
// thread, stream, completion event and accumulation buffer per device, the RGB8 frame buffer on the first device,
// and peer access from the first device to the others (enabled once).  Per frame each worker uploads the scene to
// its device (render_scene builds a new scene per call, src/main.rs:65-130) and launches the path tracer on its
// sample range; the first device then waits on the others' events (stream-ordered, no host round trip), sums all
// buffers inside the resolve (resolve_peers_kernel over NVLink peer pointers) and copies the frame out.
}  // extern "C"

struct B200rtMulti {
    struct Dev {
        int id = 0;
        cudaStream_t stream = nullptr; cudaEvent_t done = nullptr;
        float* accum = nullptr; size_t accum_bytes = 0;
        B200rtScene* scene = nullptr;
        int rc = 0; std::string err; bool ran = false;
        std::thread th;
    };
    std::vector<Dev> dv;
    uint8_t* d_rgb = nullptr; size_t rgb_bytes = 0;
    // one frame's job, published to the workers under `mu`
    std::mutex mu; std::condition_variable cv_go, cv_done;
    uint64_t generation = 0; uint32_t pending = 0; bool quit = false;
    const B200rtSceneDesc* desc = nullptr; const B200rtCamera* cam = nullptr; const B200rtRenderParams* prm = nullptr;
    std::mutex call_mu;            // one frame at a time per handle
};

namespace {

// what device k does for a frame: scene upload (+ BVH build), buffer, launch on its sample range, completion event
void multi_device_job(B200rtMulti* m, uint32_t k) {
    B200rtMulti::Dev& d = m->dv[k];
    d.rc = B200RT_OK; d.err.clear(); d.ran = false; d.scene = nullptr;
    auto bad = [&](int rc) { d.rc = rc; d.err = g_last_error; };
    if (cudaSetDevice(d.id) != cudaSuccess) { fail(B200RT_ECUDA, "cudaSetDevice(%d) failed", d.id); return bad(B200RT_ECUDA); }
    const uint32_t n = (uint32_t)m->dv.size();
    const uint32_t total = m->prm->samples == 0 ? 1 : m->prm->samples;   // src/main.rs:75-80
    const size_t px = (size_t)m->cam->image_width * m->cam->image_height;
    if (int rc = b200rt_scene_create(m->desc, d.id, &d.scene)) return bad(rc);
    if (cudaError_t e = grow(d.accum, d.accum_bytes, px * sizeof(float4))) {
        fail(B200RT_ENOMEM, "device %d: accumulation buffer: %s", d.id, cudaGetErrorString(e)); return bad(B200RT_ENOMEM);
    }
    B200rtRenderParams p = *m->prm;
    const uint32_t s0 = (uint32_t)((uint64_t)total * k / n), s1 = (uint32_t)((uint64_t)total * (k + 1) / n);
    p.flags &= ~B200RT_FLAG_ACCUMULATE; p.device = -1;
    p.sample_offset = m->prm->sample_offset + s0; p.samples = s1 - s0;
    if (s1 == s0) {   // more devices than samples: this one contributes zeros
        if (cudaMemsetAsync(d.accum, 0, px * sizeof(float4), d.stream) != cudaSuccess) { fail(B200RT_ECUDA, "memset failed"); return bad(B200RT_ECUDA); }
    } else {
        if (int rc = b200rt_render_device(d.scene, m->cam, &p, d.accum, d.stream)) return bad(rc);
        d.ran = true;
    }
    if (cudaEventRecord(d.done, d.stream) != cudaSuccess) { fail(B200RT_ECUDA, "cudaEventRecord failed"); return bad(B200RT_ECUDA); }
}

void multi_worker(B200rtMulti* m, uint32_t k) {
    uint64_t seen = 0;
    for (;;) {
        {
            std::unique_lock<std::mutex> lk(m->mu);
            m->cv_go.wait(lk, [&] { return m->quit || m->generation != seen; });
            if (m->quit) return;
            seen = m->generation;
        }
        multi_device_job(m, k);
        { std::lock_guard<std::mutex> lk(m->mu); if (--m->pending == 0) m->cv_done.notify_all(); }
    }
}

std::mutex g_multi_mu;
std::map<std::vector<int>, B200rtMulti*> g_multi_cache;    // b200rt_render_rgb8_multi: one handle per device list, for the process

}  // namespace

extern "C" {

void b200rt_multi_destroy(B200rtMulti* m) {
    if (!m) return;
    { std::lock_guard<std::mutex> lk(m->mu); m->quit = true; }
    m->cv_go.notify_all();
    for (auto& d : m->dv) if (d.th.joinable()) d.th.join();
    for (auto& d : m->dv) {
        DeviceGuard guard(d.id);
        if (d.stream) cudaStreamSynchronize(d.stream);
        if (d.accum) cudaFree(d.accum);
        if (d.done) cudaEventDestroy(d.done);
        if (d.stream) cudaStreamDestroy(d.stream);
    }
    if (m->d_rgb && !m->dv.empty()) { DeviceGuard guard(m->dv[0].id); cudaFree(m->d_rgb); }
    delete m;
}

int b200rt_multi_create(const int* devices, uint32_t n_devices, B200rtMulti** out) {
    if (!devices || !out) return fail(B200RT_EINVAL, "NULL argument");
    *out = nullptr;
    if (n_devices < 1 || n_devices > (uint32_t)MAX_PEERS) return fail(B200RT_EINVAL, "n_devices %u outside [1, %d]", n_devices, MAX_PEERS);
    for (uint32_t k = 0; k < n_devices; ++k)
        for (uint32_t j = 0; j < k; ++j) if (devices[j] == devices[k]) return fail(B200RT_EINVAL, "device %d listed twice", devices[k]);
    B200rtMulti* m = new B200rtMulti();
    m->dv.resize(n_devices);
    int rc = B200RT_OK;
    for (uint32_t k = 0; k < n_devices && rc == B200RT_OK; ++k) {
        B200rtMulti::Dev& d = m->dv[k];
        if ((rc = resolve_device(devices[k], &d.id))) break;
        DeviceGuard guard(d.id);
        cudaError_t e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.done, cudaEventDisableTiming);
        if (e != cudaSuccess) rc = fail(B200RT_ECUDA, "device %d: %s", d.id, cudaGetErrorString(e));
    }
    if (rc == B200RT_OK && n_devices > 1) {     // the first device reads every other device's buffer in the fused resolve
        DeviceGuard guard(m->dv[0].id);
        for (uint32_t k = 1; k < n_devices && rc == B200RT_OK; ++k) {
            int can = 0;
            cudaDeviceCanAccessPeer(&can, m->dv[0].id, m->dv[k].id);
            if (!can) { rc = fail(B200RT_ECUDA, "device %d cannot access device %d's memory (no peer path)", m->dv[0].id, m->dv[k].id); break; }
            cudaError_t e = cudaDeviceEnablePeerAccess(m->dv[k].id, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            if (e != cudaSuccess) rc = fail(B200RT_ECUDA, "cudaDeviceEnablePeerAccess(%d): %s", m->dv[k].id, cudaGetErrorString(e));
        }
    }
    if (rc != B200RT_OK) { std::string keep = g_last_error; b200rt_multi_destroy(m); g_last_error = keep; return rc; }
    for (uint32_t k = 1; k < n_devices; ++k) m->dv[k].th = std::thread(multi_worker, m, k);
    *out = m;
    return B200RT_OK;
}

int b200rt_multi_render_rgb8(B200rtMulti* m, const B200rtSceneDesc* desc, const B200rtCamera* cam, const B200rtRenderParams* prm,
                             uint8_t* out_rgb8, B200rtStats* stats) {
    if (!m || !desc || !cam || !prm || !out_rgb8) return fail(B200RT_EINVAL, "NULL argument");
    const size_t px = (size_t)cam->image_width * cam->image_height;
    if (px == 0) return fail(B200RT_EINVAL, "camera image dimensions are zero");
    std::lock_guard<std::mutex> call(m->call_mu);
    const uint32_t n = (uint32_t)m->dv.size();
    const uint32_t total = prm->samples == 0 ? 1 : prm->samples;
    // phase 1: every device uploads the scene and launches its sample range (workers 1..n-1; this thread is device 0)
    {
        std::lock_guard<std::mutex> lk(m->mu);
        m->desc = desc; m->cam = cam; m->prm = prm;
        m->pending = n - 1; ++m->generation;
    }
    if (n > 1) m->cv_go.notify_all();
    int prev_dev = -1; cudaGetDevice(&prev_dev);
    multi_device_job(m, 0);
    if (n > 1) { std::unique_lock<std::mutex> lk(m->mu); m->cv_done.wait(lk, [&] { return m->pending == 0; }); }
    int rc = B200RT_OK;
    for (auto& d : m->dv) if (d.rc && rc == B200RT_OK) { rc = d.rc; g_last_error = d.err; }
    // phase 2 on the first device: stream-ordered wait for everyone, fused sum + resolve over peer access, frame copy-back
    B200rtMulti::Dev& d0 = m->dv[0];
    if (rc == B200RT_OK && cudaSetDevice(d0.id) != cudaSuccess) rc = fail(B200RT_ECUDA, "cudaSetDevice(%d) failed", d0.id);
    if (rc == B200RT_OK && grow(m->d_rgb, m->rgb_bytes, px * 3) != cudaSuccess) rc = fail(B200RT_ENOMEM, "rgb8 buffer");
    if (rc == B200RT_OK) {
        const float* ptrs[MAX_PEERS];
        for (uint32_t k = 0; k < n; ++k) {
            ptrs[k] = m->dv[k].accum;
            if (k && cudaStreamWaitEvent(d0.stream, m->dv[k].done, 0) != cudaSuccess) rc = fail(B200RT_ECUDA, "cudaStreamWaitEvent failed");
        }
        if (rc == B200RT_OK) rc = b200rt_resolve_peers_rgb8_device(ptrs, n, cam->image_width, cam->image_height, total, 0, 0, m->d_rgb, nullptr, d0.stream);
        if (rc == B200RT_OK) {
            cudaError_t e = cudaMemcpyAsync(out_rgb8, m->d_rgb, px * 3, cudaMemcpyDeviceToHost, d0.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(d0.stream);
            if (e != cudaSuccess) rc = fail(B200RT_ECUDA, "frame copy-back: %s", cudaGetErrorString(e));
        }
    }
    // statistics + per-frame teardown: every device is idle once device 0's stream has drained (on an error path drain each)
    if (stats) memset(stats, 0, sizeof *stats);
    std::string keep = g_last_error;
    for (auto& d : m->dv) {
        DeviceGuard guard(d.id);
        if (rc != B200RT_OK && d.stream) cudaStreamSynchronize(d.stream);
        if (d.ran) {
            B200rtStats st{};
            if (b200rt_render_device_finish(d.scene, d.stream, &st) == B200RT_OK && stats) {
                stats->rays += st.rays; stats->paths += st.paths; stats->node_visits += st.node_visits; stats->prim_tests += st.prim_tests;
                stats->depth_exhausted += st.depth_exhausted; stats->launches += st.launches;
                stats->kernel_ms = std::max(stats->kernel_ms, st.kernel_ms); stats->total_ms = std::max(stats->total_ms, st.total_ms);
            }
        }
        if (d.scene) { b200rt_scene_destroy(d.scene); d.scene = nullptr; }
    }
    if (prev_dev >= 0) cudaSetDevice(prev_dev);
    if (rc != B200RT_OK) g_last_error = keep;
    if (stats && rc == B200RT_OK) stats->launches += 1;
    return rc;
}

// One-shot form: the handle for this device list is created on first use and kept for the life of the process
// (a host that calls render_scene once per frame pays the stream / buffer / peer-access / thread set-up once).
int b200rt_render_rgb8_multi(const B200rtSceneDesc* desc, const int* devices, uint32_t n_devices, const B200rtCamera* cam,
                             const B200rtRenderParams* prm, uint8_t* out_rgb8, B200rtStats* stats) {
    if (!desc || !devices || !cam || !prm || !out_rgb8) return fail(B200RT_EINVAL, "NULL argument");
    if (n_devices < 1 || n_devices > (uint32_t)MAX_PEERS) return fail(B200RT_EINVAL, "n_devices %u outside [1, %d]", n_devices, MAX_PEERS);
    B200rtMulti* m = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_multi_mu);
        std::vector<int> key(devices, devices + n_devices);
        auto it = g_multi_cache.find(key);
        if (it != g_multi_cache.end()) m = it->second;
        else {
            int rc = b200rt_multi_create(devices, n_devices, &m);
            if (rc) return rc;
            g_multi_cache[key] = m;
        }
    }
    return b200rt_multi_render_rgb8(m, desc, cam, prm, out_rgb8, stats);
}

int b200rt_resolve_rgb8_device(const float* d_accum, uint32_t W, uint32_t H, uint32_t samples, uint8_t* d_out, void* cuda_stream) {
    if (!d_accum || !d_out || W == 0 || H == 0) return fail(B200RT_EINVAL, "bad argument");
    dim3 block(128, 1), grid((W + 127) / 128, H);
    resolve_kernel<<<grid, block, 0, (cudaStream_t)cuda_stream>>>(reinterpret_cast<const float4*>(d_accum), W, H, samples, d_out);
    CU(cudaGetLastError());
    return B200RT_OK;
}

// ---- peer-memory buffers for the fused cross-GPU resolve -------------------------------------
int b200rt_peer_buffer_create(int device, size_t bytes, void** d_ptr, uint8_t handle[B200RT_PEER_HANDLE_BYTES]) {
    if (!d_ptr || !handle || bytes == 0) return fail(B200RT_EINVAL, "bad argument");
    static_assert(sizeof(cudaIpcMemHandle_t) <= B200RT_PEER_HANDLE_BYTES, "handle size");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    void* p = nullptr;
    CU(cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return fail(B200RT_ECUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memset(handle, 0, B200RT_PEER_HANDLE_BYTES);
    memcpy(handle, &h, sizeof h);
    CU(cudaMemset(p, 0, bytes));
    *d_ptr = p;
    return B200RT_OK;
}
int b200rt_peer_buffer_open(int device, const uint8_t handle[B200RT_PEER_HANDLE_BYTES], void** d_ptr) {
    if (!d_ptr || !handle) return fail(B200RT_EINVAL, "bad argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void* p = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) return fail(B200RT_ECUDA, "cudaIpcOpenMemHandle (is peer access between the GPUs available?): %s", cudaGetErrorString(e));
    *d_ptr = p;
    return B200RT_OK;
}
int b200rt_peer_buffer_close(int device, void* d_ptr) {
    if (!d_ptr) return B200RT_OK;
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    CU(cudaIpcCloseMemHandle(d_ptr));
    return B200RT_OK;
}
int b200rt_peer_buffer_destroy(int device, void* d_ptr) {
    if (!d_ptr) return B200RT_OK;
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    CU(cudaFree(d_ptr));
    return B200RT_OK;
}

int b200rt_peer_signal_device(uint32_t* const* d_flag_arrays, uint32_t n_peers, uint32_t my_rank, uint32_t slot, uint32_t epoch, void* cuda_stream) {
    if (!d_flag_arrays || n_peers < 1 || n_peers > (uint32_t)MAX_PEERS || my_rank >= n_peers || slot > 1) return fail(B200RT_EINVAL, "bad argument");
    PeerSignalArgs a{};
    for (uint32_t p = 0; p < n_peers; ++p) { if (!d_flag_arrays[p]) return fail(B200RT_EINVAL, "flag array %u is NULL", p); a.flags[p] = d_flag_arrays[p]; }
    a.n_peers = n_peers; a.my_rank = my_rank; a.slot = slot; a.epoch = epoch;
    peer_signal_kernel<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(a);
    CU(cudaGetLastError());
    return B200RT_OK;
}
int b200rt_peer_wait_device(uint32_t* d_my_flags, uint32_t n_peers, uint32_t slot, uint32_t epoch, uint32_t timeout_ms, void* cuda_stream) {
    if (!d_my_flags || n_peers < 1 || n_peers > (uint32_t)MAX_PEERS || slot > 1) return fail(B200RT_EINVAL, "bad argument");
    // word 2 * stride of the flag array records a time-out (1 + the rank that never arrived)
    peer_wait_kernel<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(d_my_flags, n_peers, slot, epoch, (unsigned long long)(timeout_ms ? timeout_ms : 10000) * 1000000ull,
                                                            d_my_flags + 2 * PEER_FLAG_STRIDE);
    CU(cudaGetLastError());
    return B200RT_OK;
}
int b200rt_peer_timed_out(uint32_t* d_my_flags, uint32_t* out) {
    if (!d_my_flags || !out) return fail(B200RT_EINVAL, "NULL argument");
    CU(cudaMemcpy(out, d_my_flags + 2 * PEER_FLAG_STRIDE, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (*out) CU(cudaMemset(d_my_flags + 2 * PEER_FLAG_STRIDE, 0, sizeof(uint32_t)));   // reported once: a later frame starts clean
    return B200RT_OK;
}

int b200rt_resolve_peers_rgb8_device(const float* const* d_accums, uint32_t n_peers, uint32_t W, uint32_t H, uint32_t samples,
                                     uint32_t row_begin, uint32_t row_end, uint8_t* d_out, const uint32_t* d_my_flags, void* cuda_stream) {
    if (!d_accums || !d_out || W == 0 || H == 0) return fail(B200RT_EINVAL, "bad argument");
    if (n_peers < 1 || n_peers > (uint32_t)MAX_PEERS) return fail(B200RT_EINVAL, "n_peers %u outside [1, %d]", n_peers, MAX_PEERS);
    if (row_begin == 0 && row_end == 0) row_end = H;
    if (row_end > H || row_begin > row_end) return fail(B200RT_EINVAL, "row range [%u,%u) outside image height %u", row_begin, row_end, H);
    if (row_begin == row_end) return B200RT_OK;
    PeerResolveArgs a{};
    for (uint32_t r = 0; r < n_peers; ++r) {
        if (!d_accums[r]) return fail(B200RT_EINVAL, "accumulation buffer %u is NULL", r);
        a.accum[r] = reinterpret_cast<const float4*>(d_accums[r]);
    }
    a.n_peers = n_peers; a.W = W; a.H = H; a.samples = samples; a.row_begin = row_begin; a.row_end = row_end; a.out = d_out;
    a.abort_flag = d_my_flags ? d_my_flags + 2 * PEER_FLAG_STRIDE : nullptr;    // the word peer_wait_kernel sets on a time-out
    dim3 block(128, 1), grid(((W + 3) / 4 + 127) / 128, row_end - row_begin);
    resolve_peers_kernel<<<grid, block, 0, (cudaStream_t)cuda_stream>>>(a);
    CU(cudaGetLastError());
    return B200RT_OK;
}

int b200rt_resolve_rgb8(const float* accum, uint32_t W, uint32_t H, uint32_t samples, uint8_t* out, int device) {
    if (!accum || !out || W == 0 || H == 0) return fail(B200RT_EINVAL, "bad argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    size_t px = (size_t)W * H;
    DevBuf d_acc, d_out;
    if ((rc = d_acc.alloc(px * 16)) || (rc = d_out.alloc(px * 3))) return rc;
    cudaError_t e = cudaMemcpy(d_acc.p, accum, px * 16, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) { rc = b200rt_resolve_rgb8_device(d_acc.as<float>(), W, H, samples, d_out.as<uint8_t>(), nullptr); if (rc) return rc; }
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out.p, px * 3, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(B200RT_ECUDA, "resolve: %s", cudaGetErrorString(e));
    return B200RT_OK;
}

}  // extern "C"

// ---- parity hooks ---------------------------------------------------------------------------
extern "C" {

int b200rt_closest_hit(const B200rtScene* csc, const B200rtRay* rays, size_t n, float t_min, float t_max, int32_t* ids, B200rtHit* hits, B200rtStats* stats) {
    if (!csc || (n && (!rays || !ids))) return fail(B200RT_EINVAL, "NULL argument");
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    DeviceGuard guard(sc->device);
    if (stats) memset(stats, 0, sizeof *stats);
    if (n == 0) return B200RT_OK;
    DevBuf d_rays, d_ids, d_hits, d_ctr;
    int rc;
    if ((rc = d_rays.alloc(n * sizeof(B200rtRay))) || (rc = d_ids.alloc(n * sizeof(int32_t))) || (rc = d_ctr.alloc(sizeof(Counters)))) return rc;
    if (hits && (rc = d_hits.alloc(n * sizeof(B200rtHit)))) return rc;
    CU(cudaMemcpy(d_rays.p, rays, n * sizeof(B200rtRay), cudaMemcpyHostToDevice));
    CU(cudaMemset(d_ctr.p, 0, sizeof(Counters)));
    HitArgs a{};
    a.scene = sc->ds; a.rays = d_rays.as<B200rtRay>(); a.n = n; a.t_min = t_min; a.t_max = t_max;
    a.ids = d_ids.as<int32_t>(); a.hits = hits ? d_hits.as<B200rtHit>() : nullptr; a.counters = d_ctr.as<Counters>();
    a.next_ray = &d_ctr.as<Counters>()->diag[0];     // zeroed with the counters
    const SmemPlan plan = hook_plan(scene_size(sc), sc->smem_optin);
    a.plan = plan;
    float max_origin = 0.f;
    for (size_t i = 0; i < n; ++i) max_origin = std::max(max_origin, std::max(std::fabs(rays[i].ox), std::max(std::fabs(rays[i].oy), std::fabs(rays[i].oz))));
    // traversal counters ride along with the full hit records (parity runs); ids-only calls — the BVH microbenchmark
    // shape of benches/my_benchmark.rs — run the kernel without them
    HitKernel kernel = hit_kernel(plan.all_in_smem, use_fast_slab(sc, max_origin), stats != nullptr && hits != nullptr);
    if ((rc = set_smem(kernel, sc, plan.bytes))) return rc;
    int bps = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, kernel, BLOCK, plan.bytes));
    if (bps < 1) return fail(B200RT_ECUDA, "closest_hit_kernel does not fit on an SM");
    size_t want = (n + BLOCK - 1) / BLOCK;
    uint32_t grid = (uint32_t)std::min<size_t>(want, (size_t)sc->sm_count * bps);      // persistent: one wave of CTAs
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    cudaError_t e = cudaEventRecord(e0);
    if (e == cudaSuccess) { kernel<<<grid, BLOCK, plan.bytes>>>(a); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaEventRecord(e1);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) rc = fail(B200RT_ECUDA, "closest_hit: %s", cudaGetErrorString(e));
    if (rc == B200RT_OK) {
        cudaMemcpy(ids, d_ids.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost);
        if (hits) cudaMemcpy(hits, d_hits.p, n * sizeof(B200rtHit), cudaMemcpyDeviceToHost);
        if (stats) {
            Counters c; cudaMemcpy(&c, d_ctr.p, sizeof c, cudaMemcpyDeviceToHost);
            stats->rays = c.rays; stats->node_visits = c.nodes; stats->prim_tests = c.prims; stats->launches = 1;
            float ms = 0; cudaEventElapsedTime(&ms, e0, e1); stats->kernel_ms = ms; stats->total_ms = ms;
        }
        e = cudaGetLastError();
        if (e != cudaSuccess) rc = fail(B200RT_ECUDA, "closest_hit copy-back: %s", cudaGetErrorString(e));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

int b200rt_aabb_hit(const float* boxes6, const B200rtRay* rays, size_t n, float t_min, float t_max, uint8_t* out, int device) {
    if (n && (!boxes6 || !rays || !out)) return fail(B200RT_EINVAL, "NULL argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    if (n == 0) return B200RT_OK;
    DevBuf b, r, o;
    if ((rc = b.alloc(n * 24)) || (rc = r.alloc(n * sizeof(B200rtRay))) || (rc = o.alloc(n))) return rc;
    CU(cudaMemcpy(b.p, boxes6, n * 24, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(r.p, rays, n * sizeof(B200rtRay), cudaMemcpyHostToDevice));
    aabb_hit_kernel<<<(unsigned)((n + 255) / 256), 256>>>(b.as<float>(), r.as<B200rtRay>(), n, t_min, t_max, o.as<uint8_t>());
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, o.p, n, cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_scatter(const B200rtScene* csc, const B200rtRay* rays, const B200rtHit* hits, size_t n, uint64_t seed, B200rtScatter* out) {
    if (!csc || (n && (!rays || !hits || !out))) return fail(B200RT_EINVAL, "NULL argument");
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    DeviceGuard guard(sc->device);
    if (n == 0) return B200RT_OK;
    DevBuf r, h, o; int rc;
    if ((rc = r.alloc(n * sizeof(B200rtRay))) || (rc = h.alloc(n * sizeof(B200rtHit))) || (rc = o.alloc(n * sizeof(B200rtScatter)))) return rc;
    CU(cudaMemcpy(r.p, rays, n * sizeof(B200rtRay), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(h.p, hits, n * sizeof(B200rtHit), cudaMemcpyHostToDevice));
    ScatterArgs a{}; a.scene = sc->ds; a.rays = r.as<B200rtRay>(); a.hits = h.as<B200rtHit>(); a.n = n; a.keys = rng_keys(seed); a.out = o.as<B200rtScatter>();
    scatter_kernel<<<(unsigned)((n + 127) / 128), 128>>>(a);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, o.p, n * sizeof(B200rtScatter), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_camera_rays(const B200rtCamera* cam, const float* xy, size_t n, uint64_t seed, B200rtRay* out, int device) {
    if (!cam || (n && (!xy || !out))) return fail(B200RT_EINVAL, "NULL argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    if (n == 0) return B200RT_OK;
    DevBuf x, o;
    if ((rc = x.alloc(n * 8)) || (rc = o.alloc(n * sizeof(B200rtRay)))) return rc;
    CU(cudaMemcpy(x.p, xy, n * 8, cudaMemcpyHostToDevice));
    camera_rays_kernel<<<(unsigned)((n + 255) / 256), 256>>>(make_camera(*cam), x.as<float>(), n, rng_keys(seed), o.as<B200rtRay>());
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, o.p, n * sizeof(B200rtRay), cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_texture_value(const B200rtScene* csc, int32_t tex, const float* uvp5, size_t n, float* out_rgb) {
    if (!csc || (n && (!uvp5 || !out_rgb))) return fail(B200RT_EINVAL, "NULL argument");
    B200rtScene* sc = const_cast<B200rtScene*>(csc);
    if (tex < 0 || (uint32_t)tex >= sc->ds.n_tex) return fail(B200RT_EINVAL, "texture index %d out of range", tex);
    DeviceGuard guard(sc->device);
    if (n == 0) return B200RT_OK;
    DevBuf x, o; int rc;
    if ((rc = x.alloc(n * 20)) || (rc = o.alloc(n * 12))) return rc;
    CU(cudaMemcpy(x.p, uvp5, n * 20, cudaMemcpyHostToDevice));
    TexArgs a{}; a.scene = sc->ds; a.tex = tex; a.uvp5 = x.as<float>(); a.n = n; a.out = o.as<float>();
    texture_value_kernel<<<(unsigned)((n + 127) / 128), 128>>>(a);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out_rgb, o.p, n * 12, cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_rng_uniforms(uint64_t seed, uint32_t ka, uint32_t kb, size_t n, float* out, int device) {
    if (n && !out) return fail(B200RT_EINVAL, "NULL argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    if (n == 0) return B200RT_OK;
    DevBuf o; if ((rc = o.alloc(n * 4))) return rc;
    rng_kernel<<<1, 32>>>(rng_keys(seed), ka, kb, n, o.as<float>());
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, o.p, n * 4, cudaMemcpyDeviceToHost));
    return B200RT_OK;
}

int b200rt_read_peak(int device, size_t bytes, double* gb_per_s) {
    if (!gb_per_s || bytes < (1u << 20)) return fail(B200RT_EINVAL, "bad argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    int sms = 0; CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    DevBuf b, o;
    if ((rc = b.alloc(bytes)) || (rc = o.alloc(16))) return rc;
    CU(cudaMemset(b.p, 0, bytes));
    const size_t n4 = bytes / 16;
    const int passes = (int)std::max<size_t>(2, (size_t(2) << 30) / bytes);       // ~2 GB of loads per launch
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0);
        read_peak_kernel<<<sms * 8, 256>>>(b.as<float4>(), n4, passes, o.as<float>());
        cudaEventRecord(e1);
        cudaError_t e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return fail(B200RT_ECUDA, "read_peak: %s", cudaGetErrorString(e)); }
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        if (rep > 0 && ms > 0) best = std::max(best, (double)n4 * 16.0 * passes / (ms * 1e-3) / 1e9);
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *gb_per_s = best;
    return B200RT_OK;
}

int b200rt_fp32_peak(int device, double* lane_instr_per_s) {
    if (!lane_instr_per_s) return fail(B200RT_EINVAL, "NULL argument");
    int rc = resolve_device(device, &device); if (rc) return rc;
    DeviceGuard guard(device);
    int sms = 0; CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    int grid = sms * 8, iters = 4096;
    DevBuf o; if ((rc = o.alloc((size_t)grid * 256 * 4))) return rc;
    cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 6; ++rep) {
        cudaEventRecord(e0);
        fp32_peak_kernel<<<grid, 256>>>(o.as<float>(), iters, 1.0000001f, 1e-7f);
        cudaEventRecord(e1);
        cudaError_t e = cudaEventSynchronize(e1);
        if (e != cudaSuccess) { cudaEventDestroy(e0); cudaEventDestroy(e1); return fail(B200RT_ECUDA, "fp32_peak: %s", cudaGetErrorString(e)); }
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        double ops = (double)grid * 256.0 * iters * 64.0;   // 8 chains x 8 unrolled FFMA per iteration
        if (rep > 0 && ms > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *lane_instr_per_s = best;
    return B200RT_OK;
}

}  // extern "C"
