// denoise_kernels.cuh — the feature-guided à-trous denoiser (b200rt_render_denoised, b200rt_denoise): the primary-hit feature
// pass, the conversion of the two half renders, and the filter (arithmetic in denoise_plan.hpp).
// (included by b200rt.cu; everything lives in namespace b200rt)
#pragma once
#include "denoise_plan.hpp"
#include "render_kernel.cuh"

namespace b200rt {

// ------------------------------------------------------------------------------------------
// Feature pass.  For every pixel, samples [sample_offset, sample_offset + k) of the render's own primary rays (same Rng keying,
// jitter draws and pixel_ray as path_trace_kernel_v2), traced to the first hit with the render's set-up: IEEE reciprocals,
// the up-front primitives, trav_inner_s / trav_leaf_s over the sentinel stack, the same FAST slab choice and the same staged
// (SmemAcc) or L1 (GmemAcc) scene.  Per pixel, summed over the k rays in sample order in f32 and divided by k:
//   feat[0][p] = (face-flipped normal of make_hit, t |d|)        a miss adds (0, 0, 0, 0)
//   feat[1][p] = (albedo, 0)                                     shade_prepare + marble for Lambertian and the lights, the albedo
//                                                                of Metal, (1, 1, 1) for Dielectric, background(d) for a miss
// t |d| (= |p - o|) is rounded as fl(t * fl(sqrt(fl(fl(dx dx + dy dy) + dz dz)))), so a host can reproduce it from closest_hit.
// Persistent: every CTA stages the scene once and walks blocks of blockDim.x pixels; the marble's turbulence is evaluated by
// the whole warp (coop_turbulence), so every lane runs every sample, in range or not.
// ------------------------------------------------------------------------------------------
struct FeatureArgs {
    DeviceScene scene;
    DeviceCamera cam;
    SmemPlan plan;
    RngKeys keys;
    uint32_t sample_offset, k;
    float4* feat;              // [2][H][W]
};

template <class Acc, bool FAST>
__global__ void __launch_bounds__(768, 1) denoise_feature_kernel(const __grid_constant__ FeatureArgs a) {
    extern __shared__ float4 smem[];
    int* stack_base;
    Acc acc = Stager<Acc>::stage(a.scene, a.plan, smem, &stack_base);
    int* stack = stack_base + threadIdx.x;
    stack[0] = B200RT_TRAV_DONE;
    const uint32_t stack_s = (uint32_t)__cvta_generic_to_shared(stack);
    const int stride = (int)blockDim.x * 4;
    const float T_MIN = 0.001f;                      // render.rs:31, as the render kernel
    const uint32_t n_px = a.cam.width * a.cam.height;
    for (uint32_t base = blockIdx.x * blockDim.x; base < n_px; base += gridDim.x * blockDim.x) {   // CTA-uniform
        const uint32_t pixel = base + threadIdx.x;
        const bool in_range = pixel < n_px;
        const uint32_t py = in_range ? pixel / a.cam.width : 0u, px = in_range ? pixel - py * a.cam.width : 0u;
        float4 nz = make_float4(0.f, 0.f, 0.f, 0.f), alb = make_float4(0.f, 0.f, 0.f, 0.f);
        for (uint32_t s = 0; s < a.k; ++s) {
            Rng qr;
            qr.init(a.keys, pixel, a.sample_offset + s);
            const float jx = (float)px + qr.gen();
            const float jy = (float)py + qr.gen();
            RayF ray = make_ray_shade(f3(0, 0, 0), f3(0, 0, 1));
            pixel_ray(a.cam, qr, jx, jy, &ray.o, &ray.d);
            Closest c; c.t = INFINITY; c.code = -1;
            int node = B200RT_TRAV_DONE;
            if (in_range) {
                float3 inv_e = f3(__frcp_rn(ray.d.x), __frcp_rn(ray.d.y), __frcp_rn(ray.d.z));
                ray.inv = FAST ? f3(clamp_inv(inv_e.x), clamp_inv(inv_e.y), clamp_inv(inv_e.z)) : inv_e;
                ray.nood = f3(-(ray.o.x * ray.inv.x), -(ray.o.y * ray.inv.y), -(ray.o.z * ray.inv.z));
#pragma unroll 1
                for (uint32_t t = 0; t < a.scene.n_top_prims; ++t) hit_leaf(ray, acc, a.scene.top_prims[t], T_MIN, c, &inv_e);
                node = 0;
            }
            uint32_t top = stack_s + (uint32_t)stride;
            TravCounters tc; tc.nodes = 0; tc.prims = 0;
            while (node != B200RT_TRAV_DONE) {
                if (node >= 0) trav_inner_s<false, FAST>(ray, acc, top, stride, T_MIN, c, node, tc);
                else trav_leaf_s<false>(ray, acc, top, stride, T_MIN, c, node, tc);
            }
            // ---- the shading point, warp-synchronous ----
            const bool hit = in_range && c.code >= 0;
            HitRec h; h.p = f3(0.f, 0.f, 0.f); h.n = f3(0.f, 0.f, 0.f);
            ShadePrep sp; sp.tex.need_perlin = false; sp.tex.perlin_idx = 0; sp.tex.perlin_scale = 0.f; sp.tex.rgb = f3(0.f, 0.f, 0.f);
            sp.m.kind = B200RT_MAT_LAMBERTIAN;
            if (hit) { h = make_hit(ray, acc, c); sp = shade_prepare(a.scene, acc, h); }
            const bool need = hit && sp.tex.need_perlin;
            float turb = 0.0f;
            if (a.scene.perlin != nullptr && __any_sync(0xffffffffu, need)) turb = coop_turbulence(a.scene.perlin, need, h.p, sp.tex.perlin_idx);
            float3 al = sp.tex.need_perlin ? marble(sp.tex.perlin_scale, h.p, turb) : sp.tex.rgb;
            if (hit && sp.m.kind == B200RT_MAT_METAL) al = f3(sp.m.m0.x, sp.m.m0.y, sp.m.m0.z);
            if (hit && sp.m.kind == B200RT_MAT_DIELECTRIC) al = f3(1.f, 1.f, 1.f);
            if (!hit) al = background(a.scene, ray.d);
            float depth = 0.0f;
            if (hit) {
                const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(ray.d.x, ray.d.x), __fmul_rn(ray.d.y, ray.d.y)), __fmul_rn(ray.d.z, ray.d.z)));
                depth = __fmul_rn(c.t, len);
            }
            nz.x = __fadd_rn(nz.x, h.n.x); nz.y = __fadd_rn(nz.y, h.n.y); nz.z = __fadd_rn(nz.z, h.n.z); nz.w = __fadd_rn(nz.w, depth);
            alb.x = __fadd_rn(alb.x, al.x); alb.y = __fadd_rn(alb.y, al.y); alb.z = __fadd_rn(alb.z, al.z);
        }
        if (in_range) {
            const float kf = (float)a.k;
            a.feat[pixel] = make_float4(__fdiv_rn(nz.x, kf), __fdiv_rn(nz.y, kf), __fdiv_rn(nz.z, kf), __fdiv_rn(nz.w, kf));
            a.feat[n_px + pixel] = make_float4(__fdiv_rn(alb.x, kf), __fdiv_rn(alb.y, kf), __fdiv_rn(alb.z, kf), 0.0f);
        }
    }
}

// The two half renders' fixed-point sums -> their float4 buffers and the whole render's, each with finalize_kernel's arithmetic
// ((float)sum * 2^-32, .w = the sample count): `accum` is the plain n-sample render bit for bit, and acc_a / acc_b are plain
// renders of [0, h) and [h, n) as long as no sample exceeds the 2e9 / n clamp.
__global__ void denoise_halves_kernel(const long long* __restrict__ fa, const long long* __restrict__ fb, uint32_t n_px, uint32_t na, uint32_t nb,
                                      float4* acc_a, float4* acc_b, float4* accum) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_px) return;
    const float inv = 1.0f / 4294967296.0f;
    const long long a0 = fa[p * 3 + 0], a1 = fa[p * 3 + 1], a2 = fa[p * 3 + 2];
    const long long b0 = fb[p * 3 + 0], b1 = fb[p * 3 + 1], b2 = fb[p * 3 + 2];
    acc_a[p] = make_float4((float)a0 * inv, (float)a1 * inv, (float)a2 * inv, (float)na);
    acc_b[p] = make_float4((float)b0 * inv, (float)b1 * inv, (float)b2 * inv, (float)nb);
    accum[p] = make_float4((float)(a0 + b0) * inv, (float)(a1 + b1) * inv, (float)(a2 + b2) * inv, (float)(na + nb));
}

// ------------------------------------------------------------------------------------------
// The filter: one thread per pixel, neighbours read through L1.  X = (x.rgb, v) per pixel.
// ------------------------------------------------------------------------------------------
struct FilterArgs {
    const float4* acc_a; const float4* acc_b;     // the two halves {sum rgb, count}
    const float4* feat;                           // [2][H][W]: (N, z), (albedo, 0)
    const float4* x_in; float4* x_out;
    uint32_t W, H, step;
    uint32_t last;                                // 1: remodulate and write {mean * n, n} into x_out
};

__global__ void denoise_demodulate_kernel(const __grid_constant__ FilterArgs a) {
    const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= a.W || y >= a.H) return;
    const size_t p = (size_t)y * a.W + x, n_px = (size_t)a.W * a.H;
    const float4 A = a.acc_a[p], B = a.acc_b[p], al = a.feat[n_px + p];
    const float n = A.w + B.w;
    const float ar = dn_albedo_floor(al.x), ag = dn_albedo_floor(al.y), ab = dn_albedo_floor(al.z);
    const float inv_n = n > 0.0f ? 1.0f / n : 0.0f;
    const float cr = (A.x + B.x) * inv_n, cg = (A.y + B.y) * inv_n, cb = (A.z + B.z) * inv_n;
    const float ia = A.w > 0.0f ? 1.0f / A.w : 0.0f, ib = B.w > 0.0f ? 1.0f / B.w : 0.0f;
    const float la = dn_luminance(A.x * ia / ar, A.y * ia / ag, A.z * ia / ab);
    const float lb = dn_luminance(B.x * ib / ar, B.y * ib / ag, B.z * ib / ab);
    a.x_out[p] = make_float4(cr / ar, cg / ag, cb / ab, dn_two_halves_variance(la, lb, A.w, B.w));
}

__global__ void denoise_atrous_kernel(const __grid_constant__ FilterArgs a) {
    const int x = (int)(blockIdx.x * blockDim.x + threadIdx.x), y = (int)(blockIdx.y * blockDim.y + threadIdx.y);
    const int W = (int)a.W, H = (int)a.H;
    if (x >= W || y >= H) return;
    const size_t p = (size_t)y * W + x, n_px = (size_t)W * H;
    const float4 fp = __ldg(a.feat + p), ap = __ldg(a.feat + n_px + p);
    if (fp.w == 0.0f) {                                           // the sky keeps its own sums
        if (a.last) {
            const float4 A = a.acc_a[p], B = a.acc_b[p];
            a.x_out[p] = make_float4(A.x + B.x, A.y + B.y, A.z + B.z, A.w + B.w);
        } else a.x_out[p] = a.x_in[p];
        return;
    }
    const float4 xp = __ldg(a.x_in + p);
    float vbar = 0.0f;
    for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
            const int qx = min(max(x + dx, 0), W - 1), qy = min(max(y + dy, 0), H - 1);
            vbar += dn_g3(dx) * dn_g3(dy) * __ldg(a.x_in + (size_t)qy * W + qx).w;
        }
    const float lp = dn_luminance(xp.x, xp.y, xp.z);
    const float lscale = DN_SIGMA_L * sqrtf(fmaxf(vbar, 0.0f)) + DN_EPS_L;
    const int s = (int)a.step;
    float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
    for (int dy = -2; dy <= 2; ++dy) {
        const int qy = y + dy * s;
        if (qy < 0 || qy >= H) continue;
        for (int dx = -2; dx <= 2; ++dx) {
            const int qx = x + dx * s;
            if (qx < 0 || qx >= W) continue;
            const size_t q = (size_t)qy * W + qx;
            const float4 xq = __ldg(a.x_in + q);
            float w = dn_b3(dx) * dn_b3(dy);
            if (dx != 0 || dy != 0) {
                const float4 fq = __ldg(a.feat + q), aq = __ldg(a.feat + n_px + q);
                const float dist = (float)(s * max(abs(dx), abs(dy)));
                w *= dn_edge_weight(lp, dn_luminance(xq.x, xq.y, xq.z), lscale, fp.x, fp.y, fp.z, fp.w, fq.x, fq.y, fq.z, fq.w,
                                    ap.x, ap.y, ap.z, aq.x, aq.y, aq.z, dist);
            }
            sw += w; sr += w * xq.x; sg += w * xq.y; sb += w * xq.z; sv += w * w * xq.w;
        }
    }
    const float iw = 1.0f / sw;
    float4 o = make_float4(sr * iw, sg * iw, sb * iw, sv * iw * iw);
    if (a.last) {
        const float n = a.acc_a[p].w + a.acc_b[p].w;
        o = make_float4(o.x * dn_albedo_floor(ap.x) * n, o.y * dn_albedo_floor(ap.y) * n, o.z * dn_albedo_floor(ap.z) * n, n);
    }
    a.x_out[p] = o;
}

}  // namespace b200rt
