// node_layout.hpp — the 64-byte BVH inner node the traversal reads (rt_device.cuh: BvhNode, trav_inner_s), packed from the
// builders' (lo, hi) child boxes.  Both builders call pack_node: the host SAH builder's upload (b200rt.cu) and the device
// linear BVH (lbvh.cuh: emit_kernel).  Pure arithmetic, so tests/native/node_layout_check.cpp checks it with g++.
//
// Each child box is stored as centre c and half-extent h, and each component as a (child 0, child 1) pair, so that one
// packed FP32 instruction (fma.rn.f32x2 = FFMA2 on sm_100) runs the same slab-test FMA for both children:
//   q0 = (c0.x, c1.x, c0.y, c1.y)
//   q1 = (c0.z, c1.z, h0.x, h1.x)
//   q2 = (h0.y, h1.y, h0.z, h1.z)
//   q3 = (bits(ref0), bits(ref1), 0, 0)
// i.e. float slot 2k + ch holds c[k] of child ch and slot 6 + 2k + ch its h[k].  ref >= 0: inner-node index; ref < 0: leaf,
// ~ref = (prim_type << 28) | hit_id.
#pragma once
#include <cfloat>
#include <cmath>
#include <cstring>

#ifdef __CUDACC__
#define B200RT_NL_HD __host__ __device__
#else
#define B200RT_NL_HD
#endif

namespace b200rt {

constexpr int NODE_C = 0;       // float slot of c[k] of child ch: NODE_C + 2 k + ch
constexpr int NODE_H = 6;       // float slot of h[k] of child ch: NODE_H + 2 k + ch
constexpr int NODE_REF = 12;    // float slot of bits(ref ch): NODE_REF + ch

// One axis of a child box as centre + half-extent, rounded outwards: c = (lo + hi) / 2, h = max(hi - c, c - lo) bumped up one
// ulp, so [c - h, c + h] contains [lo, hi].  An empty axis (lo > hi, or a NaN bound) gets h = -1: near > far, never entered.
// A box with an infinite bound, or one whose c or h overflows, gets c = 0, h = 3e38: always entered.
B200RT_NL_HD inline void centre_half(float lo, float hi, float* c, float* h) {
    *c = 0.f; *h = -1.f;
    if (lo <= hi) {
        *c = 0.5f * lo + 0.5f * hi;
        *h = nextafterf(fmaxf(hi - *c, *c - lo), INFINITY);
        if (!(fabsf(*c) <= FLT_MAX) || !(fabsf(*h) <= FLT_MAX)) { *c = 0.f; *h = 3.0e38f; }
    }
}

// The 16 floats of one node from the boxes (lo0, hi0) and (lo1, hi1) of its two children and their references.
B200RT_NL_HD inline void pack_node(const float lo0[3], const float hi0[3], const float lo1[3], const float hi1[3], int ref0, int ref1, float q[16]) {
    for (int k = 0; k < 3; ++k) {
        centre_half(lo0[k], hi0[k], &q[NODE_C + 2 * k], &q[NODE_H + 2 * k]);
        centre_half(lo1[k], hi1[k], &q[NODE_C + 2 * k + 1], &q[NODE_H + 2 * k + 1]);
    }
    memcpy(&q[NODE_REF], &ref0, 4);
    memcpy(&q[NODE_REF + 1], &ref1, 4);
    q[14] = 0.f; q[15] = 0.f;
}

}  // namespace b200rt
