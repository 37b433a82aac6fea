// rt_device.cuh — device-side data layout, math, RNG, intersection, traversal and shading
// for the sm_100a path tracer.  Everything here is f32.  Reference citations are relative
// to /root/reference/src/raytracer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200rt.h"
#include "launch_plan.hpp"
#include "node_layout.hpp"

namespace b200rt {

// ------------------------------------------------------------------------------------------
// Device scene layout (all arrays 16-byte aligned, read-only during a launch)
// ------------------------------------------------------------------------------------------
// BVH2 inner node, 64 B = 4 x float4 (one 16-byte vector load each); each child box is stored as
// centre c and half-extent h (the three-FMA slab test below), rounded outwards from (lo, hi), and
// each component as a (child 0, child 1) pair for the packed slab test (node_layout.hpp):
//   q0 = (c0.x, c1.x, c0.y, c1.y)
//   q1 = (c0.z, c1.z, h0.x, h1.x)
//   q2 = (h0.y, h1.y, h0.z, h1.z)
//   q3 = (bits(child0), bits(child1), 0, 0)
// child >= 0: inner-node index; child < 0: leaf, ~child = (prim_type << 28) | hit_id.
// An empty child has h = -1 (never entered), an unbounded one c = 0, h = 3e38.
// The boxes of BOTH children live in the parent, so one node fetch feeds two slab tests
// (the reference's TreeNode is 72 B of f64 per box and tests at pop, bvh/bbox_tree.rs:16-20,
// :73-76).  Nodes are stored breadth-first: the first K nodes are the top of the tree and
// are the ones staged in shared memory when the whole tree does not fit.
struct BvhNode { float4 q0, q1, q2, q3; };

#define B200RT_LEAF_TYPE_SHIFT 28
#define B200RT_LEAF_ID_MASK 0x0FFFFFFFu
// Closest::code = (type << 28) | (box face / 2 << 26) | id: the face of a RectBox hit rides in two spare bits (ids stay below 2^26)
#define B200RT_CODE_ID_MASK 0x03FFFFFFu
#define B200RT_CODE_FACE_SHIFT 26
#define B200RT_EMPTY_LEAF ((int)0x80000000)   // ~0x7FFFFFFF: never produced for a real prim

// Geometry record per hit id, 32 B = 2 x float4:
//   sphere: g0 = (cx, cy, cz, r)
//   rect:   g0 = (d1_min, d1_max, d2_min, d2_max), g1.x = offset
//   box:    g0 = (min.xyz, -), g1 = (max.xyz, -)
struct GeomRec { float4 g0, g1; };

// Material record per hit id, 32 B:
//   m0 = (r, g, b, param)   Metal: albedo + fuzz; Dielectric: param = ir;
//                           Lambertian/lights with a SOLID texture: rgb resolved at upload
//   kind = B200RT_MAT_*; tex = texture index or -1 when rgb is already resolved
struct MatRec { float4 m0; uint32_t kind; int32_t tex; uint32_t pad0, pad1; };

struct TexRec { uint32_t kind; float r, g, b; float scalar; int32_t odd, even, image; };   // 32 B

struct ImageRec { const uchar4* texels; uint32_t width, height; uint32_t pad; };
struct PerlinRec { float4 ranfloat[256]; uint8_t perm_x[256], perm_y[256], perm_z[256]; };

struct DeviceScene {
    const BvhNode* nodes;       // ONE copy of the tree, child boxes as (centre.xyz, half.xyz)
    const GeomRec* geom;
    const MatRec* mats;
    const TexRec* tex;
    const ImageRec* images;
    const PerlinRec* perlin;
    uint32_t n_nodes, n_prims, n_tex, bvh_depth, n_perlin;
    uint32_t sky_kind; float sky_r, sky_g, sky_b;
    // Primitives whose box covers most of the scene (the Weekend ground rect and its
    // dielectric coat box) are not BVH leaves: nearly every ray meets them, so they are
    // tested up front by all lanes together (no divergence) and their hit bounds the
    // traversal.  Entries are leaf-encoded (~((type << 28) | id)).  The reference keeps a
    // linear list beside its tree too (HitList for unbounded objects, scene/mod.rs:61-77).
    uint32_t n_top_prims; int top_prims[7];
    uint32_t has_emitters;      // some material is a DiffuseLight / FairyLight (else `emitted` stays zero until a path ends)
};

// Camera constants, reduced on the host in f64 from camera/mod.rs:98-114:
//   dir = llo + hw * x + vh * y - offset,   llo = lower_left - origin, hw = horizontal / W,
//   vh = vertical / H;  offset = ul * rd.x + vl * rd.y with ul = u * lens_radius.
struct DeviceCamera {
    float3 origin, llo, hw, vh, ul, vl;
    uint32_t width, height;
    int has_lens;
};


// ------------------------------------------------------------------------------------------
// Scene accessors.  The same traversal/shading code runs over a scene staged entirely in
// shared memory (SmemAcc: Weekend-sized scenes, ~60 KB, divergent 16-byte LDS cost 4
// wavefronts per warp instead of up to 32 L1 tag lookups) or resident in global memory
// behind the read-only path (GmemAcc), where the shared memory not used is left to the L1 cache.
// ------------------------------------------------------------------------------------------
struct SmemAcc {
    const float4* nodes; const float4* geom; const float4* mats; const float4* tex;
    __device__ __forceinline__ float4 node_q(int node, int k) const { return nodes[node * SMEM_NODE_QUADS + k]; }
    __device__ __forceinline__ void load_node(int node, float4& q0, float4& q1, float4& q2, float4& q3) const {
        q0 = node_q(node, 0); q1 = node_q(node, 1); q2 = node_q(node, 2); q3 = node_q(node, 3);
    }
    __device__ __forceinline__ float4 geom0(int id) const { return geom[id * 2]; }
    __device__ __forceinline__ float4 geom1(int id) const { return geom[id * 2 + 1]; }
    __device__ __forceinline__ MatRec mat(int id) const {
        float4 a = mats[id * 2], b = mats[id * 2 + 1];
        MatRec m; m.m0 = a; m.kind = __float_as_uint(b.x); m.tex = __float_as_int(b.y); m.pad0 = m.pad1 = 0; return m;
    }
    __device__ __forceinline__ TexRec texrec(int t) const {
        float4 a = tex[t * 2], b = tex[t * 2 + 1];
        TexRec T; T.kind = __float_as_uint(a.x); T.r = a.y; T.g = a.z; T.b = a.w;
        T.scalar = b.x; T.odd = __float_as_int(b.y); T.even = __float_as_int(b.z); T.image = __float_as_int(b.w); return T;
    }
};
struct GmemAcc {
    const float4* __restrict__ nodes; const float4* __restrict__ geom; const float4* __restrict__ mats; const float4* __restrict__ tex;
    // Every node comes through the read-only global path and the hardware L1.  (A staged shared-memory copy of the
    // top levels was measured: ~90 KB staged 6.4 Grays/s, 8 KB 7.3, none 7.2 on the 1e6-sphere scene — and the
    // `node < n_top` select on each of the four quads cost 15 of the 63 instructions of a traversal step.)
    // One 64-byte node = two 256-bit read-only loads (LDG.E.256 on sm_100): half the L1 requests of four 128-bit ones
    // (profiles/r02_experiments.md §15).
    __device__ __forceinline__ void load_node(int node, float4& q0, float4& q1, float4& q2, float4& q3) const {
        const float4* p = nodes + (size_t)node * 4;
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(q0.x), "=f"(q0.y), "=f"(q0.z), "=f"(q0.w), "=f"(q1.x), "=f"(q1.y), "=f"(q1.z), "=f"(q1.w) : "l"(p));
        asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                     : "=f"(q2.x), "=f"(q2.y), "=f"(q2.z), "=f"(q2.w), "=f"(q3.x), "=f"(q3.y), "=f"(q3.z), "=f"(q3.w) : "l"(p + 2));
    }
    __device__ __forceinline__ float4 geom0(int id) const { return __ldg(geom + id * 2); }
    __device__ __forceinline__ float4 geom1(int id) const { return __ldg(geom + id * 2 + 1); }
    __device__ __forceinline__ MatRec mat(int id) const {
        float4 a = __ldg(mats + id * 2), b = __ldg(mats + id * 2 + 1);
        MatRec m; m.m0 = a; m.kind = __float_as_uint(b.x); m.tex = __float_as_int(b.y); m.pad0 = m.pad1 = 0; return m;
    }
    __device__ __forceinline__ TexRec texrec(int t) const {
        float4 a = __ldg(tex + t * 2), b = __ldg(tex + t * 2 + 1);
        TexRec T; T.kind = __float_as_uint(a.x); T.r = a.y; T.g = a.z; T.b = a.w;
        T.scalar = b.x; T.odd = __float_as_int(b.y); T.even = __float_as_int(b.z); T.image = __float_as_int(b.w); return T;
    }
};

// ------------------------------------------------------------------------------------------
// float3 helpers.  Plain operators: nvcc may contract a*b+c into FMA here.  The
// intersection routines that must be reproducible bit-for-bit by oracle/gpu_f32.hpp use
// explicit __f*_rn / fmaf instead.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__device__ __forceinline__ float dot(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ float3 fma3(float s, float3 a, float3 b) { return f3(fmaf(s, a.x, b.x), fmaf(s, a.y, b.y), fmaf(s, a.z, b.z)); }
// a * b + c and a * b per component, each rounded once: ray_color's accumulators (render kernel), which the render replay
// restates on the host (tests/test_render_replay.py)
__device__ __forceinline__ float3 fma_f3(float3 a, float3 b, float3 c) { return f3(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y), fmaf(a.z, b.z, c.z)); }
__device__ __forceinline__ float3 mul_rn3(float3 a, float3 b) { return f3(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y), __fmul_rn(a.z, b.z)); }
__device__ __forceinline__ float comp(float3 a, int i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }

// ------------------------------------------------------------------------------------------
// RNG: counter-keyed PCG (documented in include/b200rt.h).  Replaces rand::ThreadRng
// (src/main.rs:98,119): a (pixel, sample) pair owns its stream, so an image does not
// depend on how tiles or sample ranges are sharded over warps or GPUs.
// ------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t pcg_out(uint32_t s) {
    uint32_t w = ((s >> ((s >> 28u) + 4u)) ^ s) * 277803737u;
    return (w >> 22u) ^ w;
}
__host__ __device__ __forceinline__ uint32_t hash32(uint32_t x) { return pcg_out(x * 747796405u + 2891336453u); }

struct RngKeys { uint32_t k0, k1; };
__host__ __device__ __forceinline__ RngKeys rng_keys(uint64_t seed) {
    RngKeys k;
    k.k0 = hash32((uint32_t)seed);
    k.k1 = hash32((uint32_t)(seed >> 32) ^ k.k0);
    return k;
}

struct Rng {
    uint32_t state, inc;
    __device__ __forceinline__ void init(RngKeys k, uint32_t a, uint32_t b) {
        state = hash32(b + hash32(a ^ k.k1));
        inc = (hash32(a + hash32(b ^ k.k0)) << 1) | 1u;
    }
    __device__ __forceinline__ uint32_t next_u32() {
        state = state * 747796405u + inc;
        return pcg_out(state);
    }
    // rng.gen::<f64>() (core/math.rs:24) at 24-bit resolution
    __device__ __forceinline__ float gen() { return (float)(next_u32() >> 8) * (1.0f / 16777216.0f); }
    // random_real(rng, -1, 1) = min + (max - min) * gen  (core/math.rs:23-25)
    // (2 g - 1 rounded once; (u >> 8) * 2^-23 - 1 in one FMA is the same value)
    __device__ __forceinline__ float gen_pm1() { return fmaf((float)(next_u32() >> 8), 1.0f / 8388608.0f, -1.0f); }
};

// ------------------------------------------------------------------------------------------
// Ray with the per-ray constants hoisted out of Aabb::hit2 (bvh/aabb.rs:66: `1.0 / d` is
// recomputed per node per axis in the reference) and Sphere::hit (sphere.rs:31: a = d.d).
// ------------------------------------------------------------------------------------------
// IEEE-rounded reciprocal, out of line: the primitive tests need it for CPU reproducibility and
// call it from several places.
__device__ __forceinline__ float rcp_exact(float x) { return __frcp_rn(x); }

struct RayF {
    float3 o, d;
    float3 inv;         // 1/d for the BOX tests only (clamped to +-1e18 for the centre-form slab test: boxes
                        // only cull and are padded).  Primitive tests take their own IEEE reciprocals so
                        // they stay bit-reproducible on the CPU.
    float3 nood;        // -(o * inv), for the one-FMA-per-plane slab test.  Stored negated so the packed slab test takes it
                        // as its addend as is: a negation written there was hoisted out of the traversal loop as three
                        // extra instructions per segment instead of being folded into FFMA2
};
__device__ __forceinline__ RayF make_ray(float3 o, float3 d) {
    RayF r;
    r.o = o; r.d = d;
    r.inv = f3(__frcp_rn(d.x), __frcp_rn(d.y), __frcp_rn(d.z));
    r.nood = f3(-(o.x * r.inv.x), -(o.y * r.inv.y), -(o.z * r.inv.z));
    return r;
}
// The slab tests take a reciprocal clamped to +-1e18: with an infinite one (direction component exactly 0) the
// one-FMA plane distance of an origin inside the slab is inf - inf = NaN on one plane and -inf on the other, which
// would cull a box the ray is inside of; a huge finite value keeps the far plane at +huge and the error analysis
// (everything scales with |inv|) unchanged.
__device__ __forceinline__ float clamp_inv(float x) { return fminf(fmaxf(x, -1e18f), 1e18f); }
// Shading-only ray (no reciprocals).
__device__ __forceinline__ RayF make_ray_shade(float3 o, float3 d) {
    RayF r;
    r.o = o; r.d = d;
    r.inv = f3(0.f, 0.f, 0.f); r.nood = r.inv;
    return r;
}

// Aabb::hit2 (bvh/aabb.rs:62-79) in f32 with the reference's exact NaN/inf behaviour:
// the swap is selected by the sign of 1/d (not by min/max of the two plane distances), a
// NaN plane distance (0 * inf) leaves the interval unchanged, `t_max <= t_min` misses.
// Returns the entry distance through *t_enter and, when asked, the exit distance through *t_exit.
__device__ __forceinline__ bool aabb_hit2(const RayF& r, float lox, float loy, float loz, float hix, float hiy, float hiz,
                                          float t_min, float t_max, float* t_enter, float* t_exit = nullptr) {
    float ax = __fmul_rn(__fsub_rn(lox, r.o.x), r.inv.x), bx = __fmul_rn(__fsub_rn(hix, r.o.x), r.inv.x);
    float ay = __fmul_rn(__fsub_rn(loy, r.o.y), r.inv.y), by = __fmul_rn(__fsub_rn(hiy, r.o.y), r.inv.y);
    float az = __fmul_rn(__fsub_rn(loz, r.o.z), r.inv.z), bz = __fmul_rn(__fsub_rn(hiz, r.o.z), r.inv.z);
    bool sx = r.inv.x < 0.0f, sy = r.inv.y < 0.0f, sz = r.inv.z < 0.0f;
    float t0x = sx ? bx : ax, t1x = sx ? ax : bx;
    float t0y = sy ? by : ay, t1y = sy ? ay : by;
    float t0z = sz ? bz : az, t1z = sz ? az : bz;
    // `if t0 > t_min {t0} else {t_min}` keeps t_min when t0 is NaN == fmaxf semantics.
    // The reference exits after each axis; the interval only ever shrinks, so testing once
    // after all three axes gives the same answer.
    float lo = fmaxf(fmaxf(t0x, t0y), fmaxf(t0z, t_min));
    float hi = fminf(fminf(t1x, t1y), fminf(t1z, t_max));
    *t_enter = lo;
    if (t_exit) *t_exit = hi;
    return !(hi <= lo);
}

// Packed FP32 FMA: (a.x * b.x + c.x, a.y * b.y + c.y), each lane rounded exactly like fmaf (fma.rn.f32x2 = one FFMA2 on
// sm_100).  A broadcast operand is passed as (s, s); ptxas folds it into the instruction's scalar operand.  The pairs are
// formed inside this one asm statement on purpose: a (s, s) pair of a ray constant packed in a statement of its own is
// loop-invariant, gets hoisted out of the traversal loop and then stays live there as an extra register pair.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t"
        ".reg .b64 a, b, c, d;\n\t"
        "mov.b64 a, {%2, %3};\n\t"
        "mov.b64 b, {%4, %5};\n\t"
        "mov.b64 c, {%6, %7};\n\t"
        "fma.rn.f32x2 d, a, b, c;\n\t"
        "mov.b64 {%0, %1}, d;\n\t"
        "}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}
// a - b and a * b per lane, rounded like __fsub_rn / __fmul_rn (FADD2 / FMUL2).
__device__ __forceinline__ float2 sub2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t"
        ".reg .b64 a, b, d;\n\t"
        "mov.b64 a, {%2, %3};\n\t"
        "mov.b64 b, {%4, %5};\n\t"
        "sub.rn.f32x2 d, a, b;\n\t"
        "mov.b64 {%0, %1}, d;\n\t"
        "}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
    float2 d;
    asm("{\n\t"
        ".reg .b64 a, b, d;\n\t"
        "mov.b64 a, {%2, %3};\n\t"
        "mov.b64 b, {%4, %5};\n\t"
        "mul.rn.f32x2 d, a, b;\n\t"
        "mov.b64 {%0, %1}, d;\n\t"
        "}"
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
    return d;
}

// Slab test on a box given as centre + half-extent: per axis
//   t_c = c * inv - o * inv,   t_near = t_c - h |inv|,   t_far = t_c + h |inv|
// — three FMAs and no min/max pair.  Against (plane - o) * inv each plane carries an extra absolute error of
// eps * |o * inv| (eps * |o| in space) plus eps * |c| for the centre; the BVH boxes are padded by more than that
// (scene_create), so a box can only be entered EARLY: the test is conservative and the closest hit unchanged.  ncu on the min/max form: the ALU pipe (FMNMX, selects,
// integer ops; half the FMA pipes' rate on sm_100) was 58 % busy against 23 % for the FMA pipes,
// with 10 ALU-pipe operations per box; this form has 4.
// Both children of a node at once, from its child-paired quads (node_layout.hpp): each of the nine FMAs is one FFMA2 over
// (child 0, child 1) with the ray constant as the broadcast operand, so each child gets exactly the bits of three scalar fmaf
// per axis.
__device__ __forceinline__ void aabb_center2(const RayF& r, float4 q0, float4 q1, float4 q2, float t_min, float t_max,
                                             float* lo0, float* hi0, float* lo1, float* hi1) {
    const float2 ix = make_float2(r.inv.x, r.inv.x), iy = make_float2(r.inv.y, r.inv.y), iz = make_float2(r.inv.z, r.inv.z);
    const float2 ox = make_float2(r.nood.x, r.nood.x), oy = make_float2(r.nood.y, r.nood.y), oz = make_float2(r.nood.z, r.nood.z);
    const float2 ax = make_float2(fabsf(r.inv.x), fabsf(r.inv.x)), ay = make_float2(fabsf(r.inv.y), fabsf(r.inv.y)),
                 az = make_float2(fabsf(r.inv.z), fabsf(r.inv.z));      // |x| is an operand modifier of FFMA2's scalar
    float2 tx = fma2(make_float2(q0.x, q0.y), ix, ox), ty = fma2(make_float2(q0.z, q0.w), iy, oy), tz = fma2(make_float2(q1.x, q1.y), iz, oz);
    float2 nx = fma2(make_float2(-q1.z, -q1.w), ax, tx), ny = fma2(make_float2(-q2.x, -q2.y), ay, ty), nz = fma2(make_float2(-q2.z, -q2.w), az, tz);
    float2 fx = fma2(make_float2(q1.z, q1.w), ax, tx), fy = fma2(make_float2(q2.x, q2.y), ay, ty), fz = fma2(make_float2(q2.z, q2.w), az, tz);
    *lo0 = fmaxf(fmaxf(nx.x, ny.x), fmaxf(nz.x, t_min)); *hi0 = fminf(fminf(fx.x, fy.x), fminf(fz.x, t_max));
    *lo1 = fmaxf(fmaxf(nx.y, ny.y), fmaxf(nz.y, t_min)); *hi1 = fminf(fminf(fx.y, fy.y), fminf(fz.y, t_max));
}

// ------------------------------------------------------------------------------------------
// Primitive intersection.  Closest-hit bookkeeping: `best_t` shrinks; the interval is
// inclusive at both ends (sphere.rs:41-46, rect.rs:58-60); among exactly equal t the
// highest hit id wins (what HitList's linear scan does, scene/mod.rs:66-76).
// These use explicit-rounding intrinsics only, so oracle/gpu_f32.hpp reproduces them
// bit-for-bit on the CPU.
// ------------------------------------------------------------------------------------------
struct Closest {
    float t;       // current closest distance (starts at t_max)
    int code;      // (type << 28) | (face / 2 << 26) | id of the closest prim, -1 = none; face (box only) = which of the 6 rects
                   // (rect.rs:149-154 order) was hit, as the first index of its pair: 0 (z), 2 (x), 4 (y)
};

__device__ __forceinline__ bool accept_t(float t, float t_min, const Closest& c, int id) {
    // NaN-safe: a NaN root is rejected.
    return (t >= t_min) && (t < c.t || (t == c.t && (c.code < 0 || id > (int)(c.code & B200RT_CODE_ID_MASK))));
}

// Sphere::hit (geometry/sphere.rs:29-52).  Same roots as the reference's textbook
// quadratic, computed in the cancellation-free form (the discriminant from the closest-
// approach vector, the roots as c/q and q/a) so that f32 stays inside 1e-5 of the f64
// reference (SURVEY.md §7).
__device__ __forceinline__ bool sphere_roots(const RayF& r, float4 s, float* root_lo, float* root_hi) {
    float ocx = __fsub_rn(r.o.x, s.x), ocy = __fsub_rn(r.o.y, s.y), ocz = __fsub_rn(r.o.z, s.z);
    float bp = -fmaf(ocz, r.d.z, fmaf(ocy, r.d.y, __fmul_rn(ocx, r.d.x)));   // -half_b
    const float a = fmaf(r.d.z, r.d.z, fmaf(r.d.y, r.d.y, __fmul_rn(r.d.x, r.d.x)));   // d.d (sphere.rs:31), taken here: one live register fewer across the traversal
    float inv_a = rcp_exact(a);
    float q = __fmul_rn(bp, inv_a);
    float lx = fmaf(q, r.d.x, ocx), ly = fmaf(q, r.d.y, ocy), lz = fmaf(q, r.d.z, ocz);
    float l2 = fmaf(lz, lz, fmaf(ly, ly, __fmul_rn(lx, lx)));
    float r2 = __fmul_rn(s.w, s.w);
    float delta = __fsub_rn(r2, l2);               // discriminant / a
    if (delta < 0.0f) return false;                // sphere.rs:35-37
    float sq = __fsqrt_rn(__fmul_rn(delta, a));  // sqrt(discriminant)
    float qq = __fadd_rn(bp, copysignf(sq, bp));
    float c = __fsub_rn(fmaf(ocz, ocz, fmaf(ocy, ocy, __fmul_rn(ocx, ocx))), r2);
    float r0 = __fdiv_rn(c, qq);
    float r1 = __fmul_rn(qq, inv_a);
    *root_lo = fminf(r0, r1);
    *root_hi = fmaxf(r0, r1);
    return true;
}

__device__ __forceinline__ void hit_sphere(const RayF& r, float4 s, int id, float t_min, Closest& c) {
    float lo, hi;
    if (!sphere_roots(r, s, &lo, &hi)) return;
    // sphere.rs:41-46: try the near root, then the far root, against [t_min, closest]
    float root = lo;
    bool ok = accept_t(root, t_min, c, id);
    if (!ok) { root = hi; ok = accept_t(root, t_min, c, id); }
    if (ok) { c.t = root; c.code = (int)((B200RT_PRIM_SPHERE << B200RT_LEAF_TYPE_SHIFT) | (uint32_t)id); }
}

// Rect<D1,D2>::hit (geometry/rect.rs:55-80) for the plane `offset` on axis dn with in-plane
// axes d1, d2.  Returns t or NaN.
// `inv_e`, when given, holds the IEEE reciprocals 1/d already taken for this ray (the render
// kernel shares them between the up-front primitives); the value is the same __frcp_rn either way.
__device__ __forceinline__ float rect_t(const RayF& r, int d1, int d2, float d1_min, float d1_max, float d2_min, float d2_max,
                                        float offset, float t_min, float t_max, const float3* inv_e = nullptr) {
    int dn = 3 - d1 - d2;
    float t = __fmul_rn(__fsub_rn(offset, comp(r.o, dn)), inv_e ? comp(*inv_e, dn) : rcp_exact(comp(r.d, dn)));
    if (!(t >= t_min && t <= t_max)) return __int_as_float(0x7fc00000);
    float a = fmaf(t, comp(r.d, d1), comp(r.o, d1));
    float b = fmaf(t, comp(r.d, d2), comp(r.o, d2));
    if (a < d1_min || a > d1_max || b < d2_min || b > d2_max) return __int_as_float(0x7fc00000);
    return t;
}

__device__ __forceinline__ void rect_axes(uint32_t type, int& d1, int& d2) {
    d1 = (type == B200RT_PRIM_RECT_YZ) ? 1 : 0;
    d2 = (type == B200RT_PRIM_RECT_XY) ? 1 : 2;
}

__device__ __forceinline__ void hit_rect(const RayF& r, uint32_t type, float4 g0, float offset, int id, float t_min, Closest& c,
                                         const float3* inv_e = nullptr) {
    int d1, d2;
    rect_axes(type, d1, d2);
    float t = rect_t(r, d1, d2, g0.x, g0.y, g0.z, g0.w, offset, t_min, c.t, inv_e);
    if (accept_t(t, t_min, c, id)) { c.t = t; c.code = (int)((type << B200RT_LEAF_TYPE_SHIFT) | (uint32_t)id); }
}

// RectBox::hit (geometry/rect.rs:147-156).  The reference takes the closest of its six
// rects, each against the shrinking interval, a later face replacing an earlier one at equal
// t (order: z faces, x faces, y faces).  A ray meets a box surface at most at its entry and
// exit points, so the same answer comes from the three slabs: the entry point if it is
// inside [t_min, closest], else the exit point; on an edge (equal t) the axis priority
// y > x > z reproduces "later replaces".  `face` records the normal axis as 0 (z), 2 (x),
// 4 (y) — the first face index of the reference's pair.
__device__ __forceinline__ void hit_box(const RayF& r, float4 lo, float4 hi, int id, float t_min, Closest& c, const float3* inv_e = nullptr) {
    float ix = inv_e ? inv_e->x : rcp_exact(r.d.x), iy = inv_e ? inv_e->y : rcp_exact(r.d.y), iz = inv_e ? inv_e->z : rcp_exact(r.d.z);
    // the x and y planes as (x, y) pairs: FADD2 + FMUL2 for the lo planes, again for the hi planes; each lane rounds as
    // __fsub_rn / __fmul_rn do, so the hit is bit for bit the scalar one
    const float2 oxy = make_float2(r.o.x, r.o.y), ixy = make_float2(ix, iy);
    const float2 axy = mul2(sub2(make_float2(lo.x, lo.y), oxy), ixy), bxy = mul2(sub2(make_float2(hi.x, hi.y), oxy), ixy);
    float ax = axy.x, ay = axy.y, bx = bxy.x, by = bxy.y;
    float az = __fmul_rn(__fsub_rn(lo.z, r.o.z), iz), bz = __fmul_rn(__fsub_rn(hi.z, r.o.z), iz);
    float nx = fminf(ax, bx), fx = fmaxf(ax, bx);
    float ny = fminf(ay, by), fy = fmaxf(ay, by);
    float nz = fminf(az, bz), fz = fmaxf(az, bz);
    float t_enter = fmaxf(fmaxf(nx, ny), nz), t_exit = fminf(fminf(fx, fy), fz);
    if (!(t_enter <= t_exit)) return;
    bool entering = t_enter >= t_min;
    float t = entering ? t_enter : t_exit;
    if (!accept_t(t, t_min, c, id)) return;
    float ty = entering ? ny : fy, tx = entering ? nx : fx;
    c.t = t;
    const uint32_t half_face = (ty == t) ? 2u : ((tx == t) ? 1u : 0u);
    c.code = (int)((B200RT_PRIM_BOX << B200RT_LEAF_TYPE_SHIFT) | (half_face << B200RT_CODE_FACE_SHIFT) | (uint32_t)id);
}

// GeometricObject::hit dispatch (geometry/object.rs:44-58)
template <class Acc>
__device__ __forceinline__ void hit_leaf(const RayF& r, const Acc& acc, int leaf, float t_min, Closest& c, const float3* inv_e = nullptr) {
    uint32_t code = (uint32_t)~leaf;
    uint32_t type = code >> B200RT_LEAF_TYPE_SHIFT;
    int id = (int)(code & B200RT_LEAF_ID_MASK);
    if (type > B200RT_PRIM_BOX) return;   // B200RT_EMPTY_LEAF
    float4 g0 = acc.geom0(id);
    if (type == B200RT_PRIM_SPHERE) {
        hit_sphere(r, g0, id, t_min, c);
    } else {
        float4 g1 = acc.geom1(id);
        if (type == B200RT_PRIM_BOX) hit_box(r, g0, g1, id, t_min, c, inv_e);
        else hit_rect(r, type, g0, g1.x, id, t_min, c, inv_e);
    }
}

// ------------------------------------------------------------------------------------------
// BVH closest-hit.  Replaces BboxTree::hit_workspace (bvh/bbox_tree.rs:56-91): instead of
// popping every child and testing its box at pop (children pushed untested, rhs first, no
// ordering), one node fetch tests both children, descends into the nearer one and pushes
// the farther one; `c.t` shrinks exactly like `t_closest`.  Closest-hit results do not
// depend on the visiting order (ties are resolved by id in accept_t).
// `stack` is a per-thread column of a shared-memory array: element k lives at
// stack[k * stride].
// ------------------------------------------------------------------------------------------
struct TravCounters { uint32_t nodes, prims; };

// ------------------------------------------------------------------------------------------
// Resumable traversal for the persistent render kernel.  The cursor (node, sp) lives in
// registers between calls so a lane can be parked while other lanes of its warp shade.
// TRAV_DONE marks "no traversal in progress".
// ------------------------------------------------------------------------------------------
#define B200RT_TRAV_DONE 0x7fffffff

// One inner-node visit: fetch the node, test both children, descend into the nearer hit child, push the farther one;
// with no hit, pop (or finish).  The stack is addressed through a moving pointer
// (`top` = next free slot of this lane's column) and its element 0 holds B200RT_TRAV_DONE, so a
// pop needs neither an index multiply nor an emptiness test: the sentinel ends the traversal.
// The step is written branch-free (selects + one predicated store / load): the three outcomes
// (both children hit / one / none) otherwise diverge inside nearly every warp step.
// With FAST slabs the whole step is 35 SASS instructions in the shared-memory render kernel and 34 in the global-memory one
// (9 FFMA2, 8 min/max, the node loads, the predicated push / pop); with one scalar FFMA per child and plane it was 44 and 42.
template <bool COUNT, bool FAST, class Acc>
__device__ __forceinline__ void trav_inner_s(const RayF& r, const Acc& acc, uint32_t& top, int stride_bytes, float t_min, const Closest& c,
                                             int& node, TravCounters& tc) {
    float4 q0, q1, q2, q3;
    acc.load_node(node, q0, q1, q2, q3);
    if (COUNT) tc.nodes++;
    float lo0, hi0, lo1, hi1;
    if (FAST) {
        aabb_center2(r, q0, q1, q2, t_min, c.t, &lo0, &hi0, &lo1, &hi1);
    } else {
        // Exact path (ray origins far outside the scene, B200RT_FAST_SLAB=0): Aabb::hit2's arithmetic on the box
        // [c - h, c + h] (a superset of the primitive's box: a box only culls).  Its verdict as an interval: a miss
        // becomes an empty one.  Child 0's c and h are the .x / .z lanes of the quads, child 1's the .y / .w lanes.
        // A single-point interval [t, t] is entered, as the centre form enters it: Aabb::hit2's `t_max <= t_min` would
        // cull it, and when the closest hit so far sits at t == t_min that drops a primitive hit at the same t with a
        // higher id (accept_t's tie rule), so the winner of the tie would depend on the visiting order.
        float e0, e1;
        aabb_hit2(r, q0.x - q1.z, q0.z - q2.x, q1.x - q2.z, q0.x + q1.z, q0.z + q2.x, q1.x + q2.z, t_min, c.t, &lo0, &e0);
        aabb_hit2(r, q0.y - q1.w, q0.w - q2.y, q1.y - q2.w, q0.y + q1.w, q0.w + q2.y, q1.y + q2.w, t_min, c.t, &lo1, &e1);
        const bool h0 = !(e0 < lo0), h1 = !(e1 < lo1);
        hi0 = h0 ? INFINITY : -INFINITY; hi1 = h1 ? INFINITY : -INFINITY;
        lo0 = h0 ? lo0 : 0.0f; lo1 = h1 ? lo1 : 0.0f;
    }
    // Three outcomes, no branch: both children hit -> push the farther, descend into the nearer;
    // one hit -> descend into it; none -> pop.  Written as PTX so the predicates stay predicates
    // (the C++ forms were compiled to select/LOP3/ISETP chains: 17-19 instructions against 13).
    int c0 = __float_as_int(q3.x), c1 = __float_as_int(q3.y), next;
    asm volatile(
        "{\n\t"
        ".reg .pred h0, h1, sw, t1, both, none;\n\t"
        ".reg .b32 far;\n\t"
        "setp.le.f32 h0, %2, %3;\n\t"
        "setp.le.f32 h1, %4, %5;\n\t"
        "setp.lt.f32 sw, %4, %2;\n\t"
        "and.pred both, h0, h1;\n\t"
        "or.pred none, h0, h1;\n\t"
        "not.pred none, none;\n\t"
        "not.pred t1, h0;\n\t"
        "or.pred t1, t1, sw;\n\t"
        "and.pred t1, t1, h1;\n\t"
        "selp.b32 %0, %7, %6, t1;\n\t"
        "selp.b32 far, %6, %7, t1;\n\t"
        "@both st.shared.b32 [%1], far;\n\t"
        "@both add.u32 %1, %1, %8;\n\t"
        "@none sub.u32 %1, %1, %8;\n\t"
        "@none ld.shared.b32 %0, [%1];\n\t"
        "}"
        : "=&r"(next), "+r"(top)
        : "f"(lo0), "f"(hi0), "f"(lo1), "f"(hi1), "r"(c0), "r"(c1), "r"(stride_bytes)
        : "memory");
    node = next;
}

template <bool COUNT, class Acc>
__device__ __forceinline__ void trav_leaf_s(const RayF& r, const Acc& acc, uint32_t& top, int stride_bytes, float t_min, Closest& c,
                                            int& node, TravCounters& tc) {
    if (COUNT) tc.prims++;
    hit_leaf(r, acc, node, t_min, c);
    top -= stride_bytes;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(node) : "r"(top) : "memory");
}

// ------------------------------------------------------------------------------------------
// Hit record (geometry/hittable.rs:17-37), built once for the winning primitive.
// ------------------------------------------------------------------------------------------
struct HitRec {
    float3 p, n;        // n is face-flipped
    float3 n_out;       // geometric (outward) normal before the flip: Sphere::get_uv input
    float t;
    bool front;
    uint32_t type; int id; int face;
    bool has_uv; float uv_u, uv_v;   // parity hooks inject the caller's (u, v); the render path computes them lazily
};

template <class Acc>
__device__ __forceinline__ HitRec make_hit(const RayF& r, const Acc& acc, const Closest& c) {
    HitRec h;
    h.has_uv = false; h.uv_u = 0.f; h.uv_v = 0.f;
    uint32_t code = (uint32_t)c.code;
    h.type = code >> B200RT_LEAF_TYPE_SHIFT;
    h.id = (int)(code & B200RT_CODE_ID_MASK);
    h.face = (int)((code >> B200RT_CODE_FACE_SHIFT) & 3u) << 1;
    h.t = c.t;
    h.p = fma3(c.t, r.d, r.o);                            // Ray::at, vec3.rs:253
    if (h.type == B200RT_PRIM_SPHERE) {
        float4 s = acc.geom0(h.id);
        float inv_r = rcp_exact(s.w);                     // sphere.rs:49 `scale(1.0 / radius)`
        // (p - center) / r, evaluated as (oc + t d) / r: one rounding instead of two
        float3 oc = f3(__fsub_rn(r.o.x, s.x), __fsub_rn(r.o.y, s.y), __fsub_rn(r.o.z, s.z));
        float3 hp = fma3(c.t, r.d, oc);
        h.n_out = f3(__fmul_rn(hp.x, inv_r), __fmul_rn(hp.y, inv_r), __fmul_rn(hp.z, inv_r));
    } else {
        int dn;
        if (h.type == B200RT_PRIM_BOX) dn = (h.face < 2) ? 2 : (h.face < 4 ? 0 : 1);
        else { int d1, d2; rect_axes(h.type, d1, d2); dn = 3 - d1 - d2; }
        h.n_out = f3(dn == 0 ? 1.0f : 0.0f, dn == 1 ? 1.0f : 0.0f, dn == 2 ? 1.0f : 0.0f);   // rect.rs:75-76
    }
    float dn_ = fmaf(r.d.z, h.n_out.z, fmaf(r.d.y, h.n_out.y, __fmul_rn(r.d.x, h.n_out.x)));
    h.front = dn_ < 0.0f;                                 // hittable.rs:25
    h.n = h.front ? h.n_out : -h.n_out;
    return h;
}

// u,v of the hit (sphere.rs:18-25, rect.rs:71-72) — only image textures read them, so they
// are computed on demand.
// Sphere::get_uv (sphere.rs:18-25), out of line: acosf + atan2f are ~200 instructions and only
// image textures need them.
__device__ __noinline__ float2 sphere_uv(float nx, float ny_, float nz) {
    const float PI = 3.14159265358979323846f;
    float ny = fminf(fmaxf(-ny_, -1.0f), 1.0f);   // f32 rounding can leave |n.y| a hair above 1
    float theta = acosf(ny);
    float phi = atan2f(-nz, nx) + PI;
    return make_float2(phi / (2.0f * PI), theta / PI);
}

template <class Acc>
__device__ __forceinline__ void hit_uv(const HitRec& h, const Acc& acc, float* u, float* v) {
    if (h.has_uv) { *u = h.uv_u; *v = h.uv_v; return; }
    if (h.type == B200RT_PRIM_SPHERE) {
        float2 uv = sphere_uv(h.n_out.x, h.n_out.y, h.n_out.z);
        *u = uv.x; *v = uv.y;
    } else {
        float4 g0; int d1, d2;
        if (h.type == B200RT_PRIM_BOX) {
            float4 lo = acc.geom0(h.id), hi = acc.geom1(h.id);
            if (h.face < 2) { d1 = 0; d2 = 1; g0 = make_float4(lo.x, hi.x, lo.y, hi.y); }
            else if (h.face < 4) { d1 = 1; d2 = 2; g0 = make_float4(lo.y, hi.y, lo.z, hi.z); }
            else { d1 = 0; d2 = 2; g0 = make_float4(lo.x, hi.x, lo.z, hi.z); }
        } else { rect_axes(h.type, d1, d2); g0 = acc.geom0(h.id); }
        float a = comp(h.p, d1), b = comp(h.p, d2);
        *u = (a - g0.x) / (g0.y - g0.x);
        *v = (b - g0.z) / (g0.w - g0.z);
    }
}

// ------------------------------------------------------------------------------------------
// Textures (material/texture/*.rs, material/perlin/mod.rs)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float perlin_noise(const PerlinRec* __restrict__ P, float3 p) {   // perlin/mod.rs:87-109
    float xf = floorf(p.x), yf = floorf(p.y), zf = floorf(p.z);
    float u = p.x - xf, v = p.y - yf, w = p.z - zf;
    int i = __float2int_rz(xf), j = __float2int_rz(yf), k = __float2int_rz(zf);   // `as i32` saturates like cvt.rzi
    float uu = u * u * (3.0f - 2.0f * u), vv = v * v * (3.0f - 2.0f * v), ww = w * w * (3.0f - 2.0f * w);   // perlin/mod.rs:43-45
    float accum = 0.0f;
#pragma unroll
    for (int di = 0; di < 2; ++di)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int dk = 0; dk < 2; ++dk) {
                int idx = P->perm_x[(i + di) & 255] ^ P->perm_y[(j + dj) & 255] ^ P->perm_z[(k + dk) & 255];
                float4 g = P->ranfloat[idx];
                float wx = u - (float)di, wy = v - (float)dj, wz = w - (float)dk;
                float blend = (di ? uu : 1.0f - uu) * (dj ? vv : 1.0f - vv) * (dk ? ww : 1.0f - ww);
                accum += blend * (g.x * wx + g.y * wy + g.z * wz);
            }
    return accum;
}

// One out-of-line copy of the accurate sine (its large-argument path is ~150 instructions and
// would otherwise be inlined four times): code size is what the instruction cache sees.
__device__ __noinline__ float sin_accurate(float x) { return sinf(x); }

// CheckerTexture::value (checker.rs:27-37) only looks at the SIGN of sin(s x) sin(s y) sin(s z):
// negative iff an odd number of the sines is negative, and sin(a) < 0 iff floor(a / pi) is odd.
// Three multiplies and floors instead of three accurate sines (arguments reach ~5e3: size 8/r
// up to 160, coordinates up to 30 — SURVEY.md §8a a17).  sin(a) is exactly 0 only at a == 0,
// where the product is +-0 and the reference takes `even`.  The cell a point falls in can
// differ from the f64 reference only within |a| * 2^-23 of a zero crossing, the same order as
// the rounding of the hit point itself.
__device__ __forceinline__ bool checker_odd(float size, float3 p) {
    const float INV_PI = 0.318309886183790671538f;
    float ax = size * p.x, ay = size * p.y, az = size * p.z;
    int k = __float2int_rd(ax * INV_PI) ^ __float2int_rd(ay * INV_PI) ^ __float2int_rd(az * INV_PI);
    bool zero = ax == 0.0f || ay == 0.0f || az == 0.0f;
    return (k & 1) && !zero;
}

// Warp-cooperative turbulence.  The marble texture costs 7 octaves x 8 lattice corners per
// evaluation, and in the Weekend scene only the few lanes that hit an odd ground cell need it
// (ncu on the per-lane loop: 2.7 of 32 lanes active).  Here the warp serves up to four requests
// per round: lane = 7 * slot + octave evaluates one full octave (perlin/mod.rs:87-109 at
// p * 2^octave, weight 2^-octave — :118-119) of the slot's request, the seven octave terms are
// summed inside each group of seven lanes and handed back to the requesting lane.  (The first
// cut spread the 56 (octave, corner) terms of ONE request over the warp: two 75-instruction
// rounds per request, 9 % of the kernel's issue slots.)  Must be called by all 32 lanes.
__device__ __noinline__ float coop_turbulence(const PerlinRec* __restrict__ tables, bool need, float3 p, int table) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int slot = (lane * 37) >> 8;                 // lane / 7 for lane < 32
    const int oct = lane - slot * 7;
    const float sc = (float)(1 << oct), wgt = 1.0f / sc;
    unsigned m = __ballot_sync(FULL, need);
    float result = 0.0f;
    while (m) {
        // the four lowest requesting lanes (a missing one repeats the first: its group's work is discarded)
        int s0 = __ffs(m) - 1;
        unsigned m1 = m & (m - 1);
        int s1 = m1 ? __ffs(m1) - 1 : s0;
        unsigned m2 = m1 & (m1 - 1);
        int s2 = m2 ? __ffs(m2) - 1 : s0;
        unsigned m3 = m2 & (m2 - 1);
        int s3 = m3 ? __ffs(m3) - 1 : s0;
        unsigned rest = m3 & (m3 - 1);
        unsigned served = m ^ rest;
        m = rest;
        int src = slot == 0 ? s0 : (slot == 1 ? s1 : (slot == 2 ? s2 : s3));
        float px = __shfl_sync(FULL, p.x, src), py = __shfl_sync(FULL, p.y, src), pz = __shfl_sync(FULL, p.z, src);
        const PerlinRec* __restrict__ P = tables + __shfl_sync(FULL, table, src);
        float v = wgt * perlin_noise(P, f3(px * sc, py * sc, pz * sc));
        float t4 = __shfl_down_sync(FULL, v, 4); if (oct < 3) v += t4;     // (0,4) (1,5) (2,6) (3)
        float t2 = __shfl_down_sync(FULL, v, 2); if (oct < 2) v += t2;     // (0,4,2,6) (1,5,3)
        float t1 = __shfl_down_sync(FULL, v, 1); if (oct < 1) v += t1;     // all seven at the group's first lane
        int rank = __popc(served & ((1u << lane) - 1u));                  // which slot served this lane's request
        float got = __shfl_sync(FULL, v, rank * 7);
        if ((served >> lane) & 1u) result = fabsf(got);
    }
    return result;
}

// Texture::value, split so the expensive marble can be evaluated cooperatively: the descent
// resolves solid / checker / image textures on the spot and returns a pending Perlin request
// otherwise.  A checker picks exactly one child per level (checker.rs:27-37), so the
// recursion is a loop.
struct TexResult { float3 rgb; bool need_perlin; int perlin_idx; float perlin_scale; };

template <class Acc>
__device__ __forceinline__ TexResult texture_descend(const Acc& acc, const ImageRec* __restrict__ images, int t, const HitRec& h) {
    TexResult out; out.rgb = f3(0.f, 0.f, 0.f); out.need_perlin = false; out.perlin_idx = 0; out.perlin_scale = 0.f;
    for (;;) {
        TexRec T = acc.texrec(t);
        if (T.kind == B200RT_TEX_SOLID) { out.rgb = f3(T.r, T.g, T.b); return out; }   // solid.rs:17-21
        if (T.kind == B200RT_TEX_CHECKER) {                                              // checker.rs:28-36
            t = checker_odd(T.scalar, h.p) ? T.odd : T.even;
            continue;
        }
        if (T.kind == B200RT_TEX_IMAGE) {                                                // image_texture.rs:34-56
            float u, v;
            hit_uv(h, acc, &u, &v);
            ImageRec im = images[T.image];
            u = fminf(fmaxf(u, 0.0f), 1.0f);
            v = 1.0f - fminf(fmaxf(v, 0.0f), 1.0f);
            uint32_t i = (uint32_t)(u * (float)(im.width - 1));     // truncation: nearest texel below, no filtering
            uint32_t j = (uint32_t)(v * (float)(im.height - 1));
            i = min(i, im.width - 1); j = min(j, im.height - 1);
            uchar4 px = __ldg(&im.texels[(size_t)j * im.width + i]);
            const float cs = 1.0f / 255.0f;
            out.rgb = f3((float)px.x * cs, (float)px.y * cs, (float)px.z * cs);
            return out;
        }
        out.need_perlin = true; out.perlin_idx = T.image; out.perlin_scale = T.scalar;
        return out;
    }
}

// Perlin marble, perlin/mod.rs:162-184: only the z lane survives the dot with (0,0,1); the
// turbulence takes the UNSCALED point (:171).
__device__ __forceinline__ float3 marble(float scale, float3 p, float turbulence) {
    float noise = 0.5f * (1.0f + sin_accurate(scale * p.z + 10.0f * turbulence));
    return f3(noise, noise, noise);
}

// ------------------------------------------------------------------------------------------
// Samplers (core/math.rs:33-81) — rejection loops in the reference's draw order
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float3 random_in_unit_sphere(Rng& rng) {   // math.rs:33-45
    for (;;) {
        float x = rng.gen_pm1(), y = rng.gen_pm1(), z = rng.gen_pm1();
        if (x * x + y * y + z * z <= 1.0f) return f3(x, y, z);
    }
}
__device__ __forceinline__ float3 unit(float3 v) {   // vec3.rs:170 (nalgebra normalize: divide by the norm)
    float inv = rsqrtf(dot(v, v));                     // MUFU.RSQ, 2 ulp: far inside the 1e-5 scatter tolerance
    return v * inv;
}

// Skybox::background (skybox/mod.rs:5-25)
__device__ __forceinline__ float3 background(const DeviceScene& s, float3 d) {
    if (s.sky_kind == B200RT_SKY_ABOVE) {
        float t = 0.5f * (d.y * rsqrtf(dot(d, d)) + 1.0f);
        return f3(1.0f - t + 0.5f * t, 1.0f - t + 0.7f * t, 1.0f);
    }
    return f3(s.sky_r, s.sky_g, s.sky_b);   // Flat(c); None is uploaded as Flat(0)
}

// Material::scatter + ::emitted (material_type.rs:50-79), in two halves around the (possibly
// cooperative) texture evaluation.  ray_color's accumulators (render.rs:24-25) are updated by the caller from what
// shade_finish returns — `emit += atten * emission` when has_emission, then `atten *= mul` when has_mul — so the
// caller decides where they live (the render kernel keeps them in shared memory: they are touched once per bounce).
// scattered == false ends the path (DiffuseLight).
struct ShadeOut { float3 o, d; float3 mul, emission; bool scattered, has_mul, has_emission; };
struct ShadePrep { MatRec m; TexResult tex; };

template <class Acc>
__device__ __forceinline__ ShadePrep shade_prepare(const DeviceScene& s, const Acc& acc, const HitRec& h) {
    ShadePrep p;
    p.m = acc.mat(h.id);
    p.tex.rgb = f3(p.m.m0.x, p.m.m0.y, p.m.m0.z);
    p.tex.need_perlin = false; p.tex.perlin_idx = 0; p.tex.perlin_scale = 0.f;
    if (p.m.tex >= 0) p.tex = texture_descend(acc, s.images, p.m.tex, h);   // Lambertian / lights with a non-solid texture
    return p;
}

__device__ __forceinline__ ShadeOut shade_finish(const RayF& r, const HitRec& h, const MatRec& m, float3 a, Rng& rng) {
    ShadeOut out;
    out.o = h.p;
    out.scattered = true;
    out.has_mul = false; out.has_emission = false;
    out.mul = f3(1.f, 1.f, 1.f); out.emission = f3(0.f, 0.f, 0.f);
    if (m.kind == B200RT_MAT_DIELECTRIC) {                              // dielectric.rs:22-49
        float ir = m.m0.w;
        float ratio = h.front ? __fdividef(1.0f, ir) : ir;   // 2-ulp divide: IEEE `/` takes its slow path for ir = 1 (0 / 2 below)
        float3 ud = unit(r.d);
        float cos_theta = fminf(-dot(ud, h.n), 1.0f);
        float sin_theta = sqrtf(1.0f - cos_theta * cos_theta);
        bool reflect = ratio * sin_theta > 1.0f;
        if (!reflect) {                                                 // `||` short-circuit: no draw under TIR
            float r0 = __fdividef(1.0f - ratio, 1.0f + ratio);
            r0 = r0 * r0;
            float k = 1.0f - cos_theta;
            float k2 = k * k;
            float refl = r0 + (1.0f - r0) * (k2 * k2 * k);              // powf(5.0), dielectric.rs:18
            reflect = refl > rng.gen();
        }
        if (reflect) {
            out.d = ud - h.n * (2.0f * dot(ud, h.n));                   // vec3.rs:135
        } else {                                                        // vec3.rs:139-145
            float3 perp = (h.n * cos_theta + ud) * ratio;
            float par = -sqrtf(fabsf(1.0f - dot(perp, perp)));
            out.d = perp + h.n * par;
        }
        return out;                                                     // attenuation = ones
    }
    if (m.kind == B200RT_MAT_DIFFUSE_LIGHT) {                           // lighting.rs:21-28
        out.emission = a; out.has_emission = true;
        out.scattered = false;
        out.d = r.d;
        return out;
    }
    // Metal, Lambertian and FairyLight all start from a point in the unit ball
    float3 rs = random_in_unit_sphere(rng);
    out.has_mul = true;
    if (m.kind == B200RT_MAT_METAL) {                                   // metal.rs:27-39: never absorbs, sampler drawn even for fuzz 0
        float3 ud = unit(r.d);
        float3 refl = ud - h.n * (2.0f * dot(ud, h.n));
        out.d = refl + rs * m.m0.w;
        out.mul = f3(m.m0.x, m.m0.y, m.m0.z);
        return out;
    }
    if (m.kind == B200RT_MAT_FAIRY_LIGHT) {                             // lighting.rs:59-66 then :43-57
        // every rounding spelled out: these are the ones nvcc chose for the render kernel from plain operators, but it
        // contracted the scatter hook's copy differently, and the hook must give the render kernel's bits
        const float nd = fmaf(h.n.z, r.d.z, fmaf(h.n.y, r.d.y, __fmul_rn(h.n.x, r.d.x)));
        const float scale = __fmul_rn(-nd, rsqrtf(fmaf(r.d.z, r.d.z, fmaf(r.d.y, r.d.y, __fmul_rn(r.d.x, r.d.x)))));
        out.emission = f3(__fmul_rn(a.x, scale), __fmul_rn(a.y, scale), __fmul_rn(a.z, scale)); out.has_emission = true;
        const float inv = rsqrtf(fmaf(a.z, a.z, fmaf(a.y, a.y, __fmul_rn(a.x, a.x))));
        a = f3(__fmul_rn(a.x, inv), __fmul_rn(a.y, inv), __fmul_rn(a.z, inv));
    }
    float3 dir = h.n + unit(rs);                                        // lambertian.rs:23, math.rs:62-68
    if (fabsf(dir.x) < 1e-8f && fabsf(dir.y) < 1e-8f && fabsf(dir.z) < 1e-8f) dir = h.n;   // vec3.rs:130
    out.d = dir;
    out.mul = a;
    return out;
}

// Camera::pixel_ray (camera/mod.rs:98-131); x, y are the jittered pixel coordinates.
__device__ __forceinline__ void pixel_ray(const DeviceCamera& cam, Rng& rng, float x, float y, float3* o, float3* d) {
    float3 offset = f3(0.0f, 0.0f, 0.0f);
    if (cam.has_lens) {                                                 // math.rs:70-81 random_in_unit_disk
        float rx, ry;
        do { rx = rng.gen_pm1(); ry = rng.gen_pm1(); } while (!(rx * rx + ry * ry <= 1.0f));
        offset = cam.ul * rx + cam.vl * ry;
    }
    *d = fma3(y, cam.vh, fma3(x, cam.hw, cam.llo)) - offset;
    *o = cam.origin + offset;
}

}  // namespace b200rt
