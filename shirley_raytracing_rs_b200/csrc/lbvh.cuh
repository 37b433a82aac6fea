// lbvh.cuh — K5: BVH construction on the device for large scenes.
//
// Replaces bvh/bbox_tree/constructor.rs:9-212 (host-side, O(N^2), degenerate beyond a few
// thousand objects — SURVEY.md §8a a24) when a scene has 1e5-1e6 primitives and the host SAH
// builder (bvh_build.hpp, ~0.5 s per 1e6 spheres on 8 threads) would dominate a frame that
// renders in tens of milliseconds on several GPUs.  Linear BVH after Karras 2012 ("Maximizing
// Parallelism in the Construction of BVHs, Octrees, and k-d Trees"):
//   1. 63-bit Morton key of every primitive's box centre (21 bits per axis over the scene's bounding cube)
//   2. radix sort of (key, primitive) pairs                      (cub::DeviceRadixSort)
//   3. one thread per internal node finds its key range and split -> children, parents
//   4. bottom-up refit: the second thread to arrive at a node (atomic counter) joins its
//      children's boxes and depths and climbs on
//   5. one thread per internal node emits the 64-byte traversal node (node_layout.hpp: pack_node)
// Closest-hit results do not depend on the tree (ties are resolved by hit id), so parity is
// unaffected; on the config-4 scene the tree costs 2 % more node visits than the SAH one (profiles/).
#pragma once
#include <cub/device/device_radix_sort.cuh>
#include <cuda_runtime.h>
#include <stdint.h>

#include "bvh_build.hpp"
#include "rt_device.cuh"

namespace b200rt {
namespace lbvh {

struct PrimBox { float4 lo, hi; };   // lo.w = bits(code), code = (type << 28) | hit id

__device__ __forceinline__ unsigned long long spread21(unsigned long long v) {   // 21 bits -> every third bit
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

__global__ void morton_kernel(const PrimBox* __restrict__ prims, uint32_t n, float3 lo, float3 inv_ext, unsigned long long* keys, uint32_t* vals) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    PrimBox b = prims[i];
    float cx = (0.5f * (b.lo.x + b.hi.x) - lo.x) * inv_ext.x, cy = (0.5f * (b.lo.y + b.hi.y) - lo.y) * inv_ext.y, cz = (0.5f * (b.lo.z + b.hi.z) - lo.z) * inv_ext.z;
    const float S = 2097151.0f;   // 2^21 - 1
    unsigned long long x = (unsigned long long)fminf(fmaxf(cx * S, 0.0f), S), y = (unsigned long long)fminf(fmaxf(cy * S, 0.0f), S),
                       z = (unsigned long long)fminf(fmaxf(cz * S, 0.0f), S);
    keys[i] = (spread21(x) << 2) | (spread21(y) << 1) | spread21(z);
    vals[i] = i;
}

// Length of the common prefix of keys i and j (ties broken by position, so all keys are distinct)
__device__ __forceinline__ int delta(const unsigned long long* __restrict__ keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    unsigned long long a = keys[i], b = keys[j];
    return a == b ? 64 + __clz(i ^ j) : __clzll((long long)(a ^ b));
}

// Child reference convention inside the builder: >= 0 internal node, < 0 ~leaf position (sorted order)
__global__ void hierarchy_kernel(const unsigned long long* __restrict__ keys, int n, int2* children, int* parent_internal, int* parent_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    int gamma = i + s * d + min(d, 0);
    int lo = min(i, j), hi = max(i, j);
    int left = lo == gamma ? ~gamma : gamma;
    int right = hi == gamma + 1 ? ~(gamma + 1) : gamma + 1;
    children[i] = make_int2(left, right);
    if (left >= 0) parent_internal[left] = i; else parent_leaf[gamma] = i;
    if (right >= 0) parent_internal[right] = i; else parent_leaf[gamma + 1] = i;
    if (i == 0) parent_internal[0] = -1;
}

struct SubBox { float lo[3], hi[3]; uint32_t depth, pad; };   // box and height of an internal node's subtree

__device__ __forceinline__ void child_box(int c, const PrimBox* __restrict__ prims, const uint32_t* __restrict__ order, const volatile SubBox* sub,
                                          float* lo, float* hi, uint32_t* depth) {
    if (c < 0) {
        PrimBox b = prims[order[~c]];
        lo[0] = b.lo.x; lo[1] = b.lo.y; lo[2] = b.lo.z; hi[0] = b.hi.x; hi[1] = b.hi.y; hi[2] = b.hi.z; *depth = 0;
    } else {
        for (int k = 0; k < 3; ++k) { lo[k] = sub[c].lo[k]; hi[k] = sub[c].hi[k]; }
        *depth = sub[c].depth;
    }
}

__global__ void refit_kernel(const PrimBox* __restrict__ prims, const uint32_t* __restrict__ order, int n, const int2* __restrict__ children,
                             const int* __restrict__ parent_internal, const int* __restrict__ parent_leaf, SubBox* sub, unsigned int* arrived) {
    int leaf = blockIdx.x * blockDim.x + threadIdx.x;
    if (leaf >= n) return;
    int node = parent_leaf[leaf];
    while (node >= 0) {
        __threadfence();                                   // publish what this thread wrote below before the counter moves
        if (atomicAdd(&arrived[node], 1u) == 0u) return;   // first arrival: the sibling subtree is not done yet
        __threadfence();
        int2 c = children[node];
        float l0[3], h0[3], l1[3], h1[3]; uint32_t d0, d1;
        child_box(c.x, prims, order, sub, l0, h0, &d0);
        child_box(c.y, prims, order, sub, l1, h1, &d1);
        for (int k = 0; k < 3; ++k) { sub[node].lo[k] = fminf(l0[k], l1[k]); sub[node].hi[k] = fmaxf(h0[k], h1[k]); }
        sub[node].depth = 1u + max(d0, d1);
        node = parent_internal[node];
    }
}

__global__ void emit_kernel(const PrimBox* __restrict__ prims, const uint32_t* __restrict__ order, int n, const int2* __restrict__ children,
                            const SubBox* __restrict__ sub, BvhNode* nodes) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int2 c = children[i];
    float l0[3], h0[3], l1[3], h1[3]; uint32_t d0, d1;
    child_box(c.x, prims, order, sub, l0, h0, &d0);
    child_box(c.y, prims, order, sub, l1, h1, &d1);
    int r0 = c.x >= 0 ? c.x : ~__float_as_int(prims[order[~c.x]].lo.w);   // leaf: ~((type << 28) | id)
    int r1 = c.y >= 0 ? c.y : ~__float_as_int(prims[order[~c.y]].lo.w);
    float q[16];
    pack_node(l0, h0, l1, h1, r0, r1, q);
    nodes[i] = BvhNode{make_float4(q[0], q[1], q[2], q[3]), make_float4(q[4], q[5], q[6], q[7]), make_float4(q[8], q[9], q[10], q[11]),
                       make_float4(q[12], q[13], q[14], q[15])};
}

// Builds the tree of `prims` (host array, boxes already padded; at least 2 entries) into
// d_nodes (n - 1 nodes in the centre/half-extent form, root = 0).  Returns a cudaError_t; *depth_out = the
// largest number of inner nodes on a root-to-leaf path.
inline cudaError_t build(const std::vector<BuildPrim>& prims, const HostBox& bounds, BvhNode* d_nodes, uint32_t* depth_out, float* build_ms) {
    const int n = (int)prims.size();
    std::vector<PrimBox> hp(n);
    for (int i = 0; i < n; ++i) {
        const BuildPrim& p = prims[i];
        float codef; int code = p.code; memcpy(&codef, &code, 4);
        hp[i].lo = make_float4(p.box.lo[0], p.box.lo[1], p.box.lo[2], codef);
        hp[i].hi = make_float4(p.box.hi[0], p.box.hi[1], p.box.hi[2], 0.f);
    }
    // one scratch allocation carved into the builder's arrays (a dozen cudaMalloc/cudaFree pairs cost more than the build)
    size_t tmp_bytes = 0;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, n, 0, 63);
    if (e != cudaSuccess) return e;
    size_t off = 0;
    auto carve = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
    const size_t o_prims = carve((size_t)n * sizeof(PrimBox)), o_keys = carve((size_t)n * 8), o_keys2 = carve((size_t)n * 8), o_vals = carve((size_t)n * 4),
                 o_vals2 = carve((size_t)n * 4), o_children = carve((size_t)(n - 1) * sizeof(int2)), o_pi = carve((size_t)(n - 1) * 4), o_pl = carve((size_t)n * 4),
                 o_sub = carve((size_t)(n - 1) * sizeof(SubBox)), o_arr = carve((size_t)(n - 1) * 4), o_tmp = carve(tmp_bytes);
    uint8_t* base = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    auto cleanup = [&]() { cudaFree(base); if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); };
#define LBVH_TRY(x) do { e = (x); if (e != cudaSuccess) { cleanup(); return e; } } while (0)
    LBVH_TRY(cudaMalloc(&base, off));
    PrimBox* d_prims = reinterpret_cast<PrimBox*>(base + o_prims);
    unsigned long long *d_keys = reinterpret_cast<unsigned long long*>(base + o_keys), *d_keys2 = reinterpret_cast<unsigned long long*>(base + o_keys2);
    uint32_t *d_vals = reinterpret_cast<uint32_t*>(base + o_vals), *d_vals2 = reinterpret_cast<uint32_t*>(base + o_vals2);
    int2* d_children = reinterpret_cast<int2*>(base + o_children);
    int *d_pi = reinterpret_cast<int*>(base + o_pi), *d_pl = reinterpret_cast<int*>(base + o_pl);
    SubBox* d_sub = reinterpret_cast<SubBox*>(base + o_sub);
    unsigned int* d_arr = reinterpret_cast<unsigned int*>(base + o_arr);
    void* d_tmp = base + o_tmp;
    LBVH_TRY(cudaMemcpy(d_prims, hp.data(), (size_t)n * sizeof(PrimBox), cudaMemcpyHostToDevice));
    LBVH_TRY(cudaEventCreate(&e0)); LBVH_TRY(cudaEventCreate(&e1));
    LBVH_TRY(cudaEventRecord(e0));
    LBVH_TRY(cudaMemsetAsync(d_arr, 0, (size_t)(n - 1) * 4));
    float3 lo = make_float3(bounds.lo[0], bounds.lo[1], bounds.lo[2]);
    // one scale for all three axes (Morton cells are cubes): a flat scene — spheres resting on a plane — must
    // not spend a third of its key bits on its thin axis (per-axis scaling: 3.4x the node visits)
    float ext = std::max(bounds.hi[0] - bounds.lo[0], std::max(bounds.hi[1] - bounds.lo[1], bounds.hi[2] - bounds.lo[2]));
    float inv1 = ext > 0.f ? 1.0f / ext : 0.f;
    float3 inv_ext = make_float3(inv1, inv1, inv1);
    const int T = 256;
    morton_kernel<<<(n + T - 1) / T, T>>>(d_prims, (uint32_t)n, lo, inv_ext, d_keys, d_vals);
    LBVH_TRY(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_vals, d_vals2, n, 0, 63));
    hierarchy_kernel<<<(n - 1 + T - 1) / T, T>>>(d_keys2, n, d_children, d_pi, d_pl);
    refit_kernel<<<(n + T - 1) / T, T>>>(d_prims, d_vals2, n, d_children, d_pi, d_pl, d_sub, d_arr);
    emit_kernel<<<(n - 1 + T - 1) / T, T>>>(d_prims, d_vals2, n, d_children, d_sub, d_nodes);
    LBVH_TRY(cudaGetLastError());
    LBVH_TRY(cudaEventRecord(e1));
    SubBox root;
    LBVH_TRY(cudaMemcpy(&root, d_sub, sizeof(SubBox), cudaMemcpyDeviceToHost));
    *depth_out = root.depth;
    if (build_ms) LBVH_TRY(cudaEventElapsedTime(build_ms, e0, e1));
#undef LBVH_TRY
    cleanup();
    return cudaSuccess;
}

}  // namespace lbvh
}  // namespace b200rt
