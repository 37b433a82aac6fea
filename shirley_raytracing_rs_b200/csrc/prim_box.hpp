// prim_box.hpp — a primitive's BVH box from its geometry record, whether it gets a leaf, the box padding, and the refit of a
// tree's boxes over the emitted node array of either builder.  b200rt_scene_create computes every leaf box with these
// functions, and b200rt_scene_update's device refit (refit.cuh) recomputes them with the same ones, so the two cannot drift.
// Pure arithmetic; tests/native/refit_check.cpp compiles it with g++ and uses refit_host as the reference of the device refit.
#pragma once
#include <cmath>
#include <cstdint>
#include <vector>

#include "../../include/b200rt.h"
#include "node_layout.hpp"

namespace b200rt {

// The box of a primitive from its geometry record (rt_device.cuh: GeomRec; F4 is float4 or any struct with x, y, z, w):
//   sphere: g0 = (cx, cy, cz, r)                             sphere.rs:54-60, centre -/+ (r, r, r); r < 0 inverts the box
//   rect:   g0 = (d1_min, d1_max, d2_min, d2_max), g1.x = k  rect.rs:9,82-99, k -/+ 0.0001 on the normal axis
//   box:    g0 = min, g1 = max                               rect.rs:158-163
template <class F4>
B200RT_NL_HD inline void prim_box(uint32_t type, const F4& g0, const F4& g1, float lo[3], float hi[3]) {
    if (type == B200RT_PRIM_SPHERE) {
        lo[0] = g0.x - g0.w; lo[1] = g0.y - g0.w; lo[2] = g0.z - g0.w;
        hi[0] = g0.x + g0.w; hi[1] = g0.y + g0.w; hi[2] = g0.z + g0.w;
    } else if (type == B200RT_PRIM_BOX) {
        lo[0] = g0.x; lo[1] = g0.y; lo[2] = g0.z;
        hi[0] = g1.x; hi[1] = g1.y; hi[2] = g1.z;
    } else {
        const int d1 = type == B200RT_PRIM_RECT_YZ ? 1 : 0, d2 = type == B200RT_PRIM_RECT_XY ? 1 : 2, dn = 3 - d1 - d2;
        lo[d1] = g0.x; hi[d1] = g0.y; lo[d2] = g0.z; hi[d2] = g0.w;
        lo[dn] = g1.x - 0.0001f; hi[dn] = g1.x + 0.0001f;
    }
}

// The reference keeps inverted boxes in its tree, where Aabb::hit2 can never pass; here they get no leaf.  NaN boxes likewise.
B200RT_NL_HD inline bool box_valid(const float lo[3], const float hi[3]) { return lo[0] <= hi[0] && lo[1] <= hi[1] && lo[2] <= hi[2]; }

B200RT_NL_HD inline float box_max_abs(const float lo[3], const float hi[3]) {
    float m = 0.f;
    for (int k = 0; k < 3; ++k) m = fmaxf(m, fmaxf(fabsf(lo[k]), fabsf(hi[k])));
    return m;
}

// Every leaf box is grown by 4e-6 x the scene's largest coordinate of a valid box (~34 ulp): the f32 slab tests are then
// conservative with respect to the f32 primitive tests (b200rt.cu, launch_plan.hpp: fast_slab_ok).  A box only culls.
B200RT_NL_HD inline float box_pad_for(float max_abs) { return max_abs * 4e-6f; }
B200RT_NL_HD inline void pad_box(float lo[3], float hi[3], float pad) { for (int k = 0; k < 3; ++k) { lo[k] -= pad; hi[k] += pad; } }

// A child box exactly as the builders hold it before packing: the union of its subtree's padded leaf boxes by f32 min / max.
struct ExactBox { float lo[3], hi[3]; };
B200RT_NL_HD inline void box_empty(ExactBox& b) { for (int k = 0; k < 3; ++k) { b.lo[k] = INFINITY; b.hi[k] = -INFINITY; } }
B200RT_NL_HD inline void box_union(ExactBox& b, const ExactBox& a, const ExactBox& c) {
    for (int k = 0; k < 3; ++k) { b.lo[k] = fminf(a.lo[k], c.lo[k]); b.hi[k] = fmaxf(a.hi[k], c.hi[k]); }
}

// Child references (node_layout.hpp): >= 0 an inner node, < 0 a leaf with ~ref = (type << 28) | hit id, or an empty slot.
constexpr int EMPTY_CHILD = (int)0x80000000;   // a child slot with no subtree (trees of 0 or 1 leaves), rt_device.cuh: B200RT_EMPTY_LEAF
constexpr uint32_t LEAF_TYPE_SHIFT = 28, LEAF_ID_MASK = 0x0FFFFFFFu;

// Links of node `i` with child references (ref0, ref1), the order-free part of the refit: parent[c] = 2 i + side for an inner
// child c, leaf_slot[hit id] = 2 i + side for a leaf.  Entries that no node sets stay -1 (the root's parent; primitives
// without a leaf: invalid boxes and the up-front list).  Both the breadth-first host tree and the Karras-numbered device tree
// are described by their child references alone.
B200RT_NL_HD inline void node_links(int i, int ref0, int ref1, int* parent, int* leaf_slot) {
    const int refs[2] = {ref0, ref1};
    for (int s = 0; s < 2; ++s) {
        const int r = refs[s];
        if (r >= 0) parent[r] = 2 * i + s;
        else if (r != EMPTY_CHILD) leaf_slot[(uint32_t)~r & LEAF_ID_MASK] = 2 * i + s;
    }
}

B200RT_NL_HD inline int node_ref(const float* q, int side) { int r; memcpy(&r, &q[NODE_REF + side], 4); return r; }

// Host twin of the device refit (refit.cuh): a post-order walk from the root that recomputes every node from the geometry
// records with the functions above.  `nodes` holds n_nodes x 16 floats in the node_layout.hpp form; G has members g0, g1 as
// GeomRec does.
template <class G>
struct HostRefit {
    float* nodes; const G* geom; float pad;
    ExactBox walk(int i) {
        float* q = nodes + 16 * (size_t)i;
        ExactBox b[2];
        for (int s = 0; s < 2; ++s) {
            const int r = node_ref(q, s);
            if (r >= 0) b[s] = walk(r);
            else if (r == EMPTY_CHILD) box_empty(b[s]);
            else {
                const uint32_t code = (uint32_t)~r, id = code & LEAF_ID_MASK;
                prim_box(code >> LEAF_TYPE_SHIFT, geom[id].g0, geom[id].g1, b[s].lo, b[s].hi);
                pad_box(b[s].lo, b[s].hi, pad);
            }
        }
        pack_node(b[0].lo, b[0].hi, b[1].lo, b[1].hi, node_ref(q, 0), node_ref(q, 1), q);
        ExactBox u; box_union(u, b[0], b[1]);
        return u;
    }
};
template <class G>
inline void refit_host(float* nodes, uint32_t n_nodes, const G* geom, float pad) {
    if (n_nodes) HostRefit<G>{nodes, geom, pad}.walk(0);
}

inline void refit_links_host(const float* nodes, uint32_t n_nodes, uint32_t n_prims, std::vector<int>* parent, std::vector<int>* leaf_slot) {
    parent->assign(n_nodes, -1);
    leaf_slot->assign(n_prims, -1);
    for (uint32_t i = 0; i < n_nodes; ++i) node_links((int)i, node_ref(nodes + 16 * (size_t)i, 0), node_ref(nodes + 16 * (size_t)i, 1), parent->data(), leaf_slot->data());
}

}  // namespace b200rt
