// refit.cuh — K6: the BVH refit of b200rt_scene_update.  The tree keeps its topology (either builder's emitted node array:
// breadth-first from the host SAH builder, Karras-numbered from the device LBVH, so nothing here assumes an order) and its
// boxes are recomputed from the new geometry records:
//   1. refit_links_kernel, once per scene: each node's parent (node, side) and each hit id's leaf slot (node, side), from the
//      child references alone (prim_box.hpp: node_links)
//   2. refit_kernel, per update: one thread per hit id computes its padded leaf box (prim_box.hpp, the functions
//      b200rt_scene_create uses); the second thread to arrive at a node (atomic counter, as lbvh.cuh: refit_kernel) unions the
//      two exact (lo, hi) child boxes, packs the node with pack_node and climbs on.
// Boxes are carried as exact (lo, hi) pairs, never unpacked from the centre/half-extent node, so an unchanged scene refits to
// the builder's nodes byte for byte and repeated updates never grow a box.  prim_box.hpp: refit_host is the host twin.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "prim_box.hpp"
#include "rt_device.cuh"

namespace b200rt {
namespace refit {

// prim_box.hpp restates these so that g++ can compile it without the CUDA headers; they must agree with the traversal's
static_assert(EMPTY_CHILD == B200RT_EMPTY_LEAF, "empty child reference");
static_assert(LEAF_TYPE_SHIFT == B200RT_LEAF_TYPE_SHIFT && LEAF_ID_MASK == B200RT_LEAF_ID_MASK, "leaf reference encoding");

__global__ void refit_links_kernel(const BvhNode* __restrict__ nodes, uint32_t n_nodes, int* parent, int* leaf_slot) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const float4 q3 = nodes[i].q3;
    node_links((int)i, __float_as_int(q3.x), __float_as_int(q3.y), parent, leaf_slot);
}

// box[2 node + side] = the exact box of that child, written by the thread that finished the child (or by its leaf's thread)
__global__ void refit_kernel(BvhNode* nodes, const GeomRec* __restrict__ geom, uint32_t n_prims, const int* __restrict__ parent,
                             const int* __restrict__ leaf_slot, ExactBox* box, unsigned int* arrived, float pad) {
    const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
    if (id >= n_prims) return;
    int slot = leaf_slot[id];
    if (slot < 0) return;                                  // no leaf: an invalid box or an up-front primitive
    int node = slot >> 1;
    ExactBox b;
    {
        const float4 q3 = nodes[node].q3;
        const uint32_t code = ~(uint32_t)__float_as_int((slot & 1) ? q3.y : q3.x);
        const GeomRec g = geom[id];
        prim_box(code >> LEAF_TYPE_SHIFT, g.g0, g.g1, b.lo, b.hi);
        pad_box(b.lo, b.hi, pad);
    }
    volatile ExactBox* vbox = box;
    while (true) {
        for (int k = 0; k < 3; ++k) { vbox[slot].lo[k] = b.lo[k]; vbox[slot].hi[k] = b.hi[k]; }
        const float4 q3 = nodes[node].q3;
        const int r0 = __float_as_int(q3.x), r1 = __float_as_int(q3.y);
        __threadfence();                                   // publish the box above before the counter moves
        if (r0 != EMPTY_CHILD && r1 != EMPTY_CHILD && atomicAdd(&arrived[node], 1u) == 0u) return;   // the sibling is not done yet
        __threadfence();
        ExactBox c[2];
        for (int s = 0; s < 2; ++s) {
            if ((s ? r1 : r0) == EMPTY_CHILD) { box_empty(c[s]); continue; }
            for (int k = 0; k < 3; ++k) { c[s].lo[k] = vbox[2 * node + s].lo[k]; c[s].hi[k] = vbox[2 * node + s].hi[k]; }
        }
        float q[16];
        pack_node(c[0].lo, c[0].hi, c[1].lo, c[1].hi, r0, r1, q);
        nodes[node] = BvhNode{make_float4(q[0], q[1], q[2], q[3]), make_float4(q[4], q[5], q[6], q[7]), make_float4(q[8], q[9], q[10], q[11]),
                              make_float4(q[12], q[13], q[14], q[15])};
        box_union(b, c[0], c[1]);
        slot = parent[node];
        if (slot < 0) return;                              // the root
        node = slot >> 1;
    }
}

// The refit's device state, allocated by the first update of a scene and kept with it: links (parent per node, leaf slot per hit
// id), the exact child boxes and the arrival counters.
struct State {
    void* base = nullptr;
    int* parent = nullptr; int* leaf_slot = nullptr; ExactBox* box = nullptr; unsigned int* arrived = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_h2d = nullptr, ev0 = nullptr, ev1 = nullptr;   // before the update's copies, around the refit kernel
    void release() {
        if (base) cudaFree(base);
        if (ev_h2d) cudaEventDestroy(ev_h2d);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (stream) cudaStreamDestroy(stream);
        *this = State{};
    }
    // allocates and derives the links; on failure nothing is kept
    cudaError_t init(const BvhNode* nodes, uint32_t n_nodes, uint32_t n_prims) {
        size_t off = 0;
        auto carve = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
        const size_t o_parent = carve((size_t)n_nodes * 4), o_leaf = carve((size_t)n_prims * 4), o_box = carve((size_t)n_nodes * 2 * sizeof(ExactBox)),
                     o_arr = carve((size_t)n_nodes * 4);
        cudaError_t e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaEventCreate(&ev_h2d);
        if (e == cudaSuccess) e = cudaEventCreate(&ev0);
        if (e == cudaSuccess) e = cudaEventCreate(&ev1);
        if (e == cudaSuccess) e = cudaMalloc(&base, off);
        if (e != cudaSuccess) { release(); return e; }
        uint8_t* p = static_cast<uint8_t*>(base);
        parent = reinterpret_cast<int*>(p + o_parent); leaf_slot = reinterpret_cast<int*>(p + o_leaf);
        box = reinterpret_cast<ExactBox*>(p + o_box); arrived = reinterpret_cast<unsigned int*>(p + o_arr);
        e = cudaMemsetAsync(parent, 0xFF, (size_t)n_nodes * 4, stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(leaf_slot, 0xFF, (size_t)n_prims * 4, stream);
        if (e == cudaSuccess && n_nodes) {
            refit_links_kernel<<<(n_nodes + 255) / 256, 256, 0, stream>>>(nodes, n_nodes, parent, leaf_slot);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) release();
        return e;
    }
    // enqueues the refit on `stream` (ev0, ev1 around the kernel)
    cudaError_t run(BvhNode* nodes, uint32_t n_nodes, const GeomRec* geom, uint32_t n_prims, float pad) {
        cudaError_t e = cudaMemsetAsync(arrived, 0, (size_t)n_nodes * 4, stream);
        if (e == cudaSuccess) e = cudaEventRecord(ev0, stream);
        if (e == cudaSuccess && n_prims) {
            refit_kernel<<<(n_prims + 255) / 256, 256, 0, stream>>>(nodes, geom, n_prims, parent, leaf_slot, box, arrived, pad);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaEventRecord(ev1, stream);
        return e;
    }
};

}  // namespace refit
}  // namespace b200rt
