"""Renders bit for bit against their paths replayed bounce by bounce through the parity hooks (DESIGN.md §4, level 4).

For every selected (pixel p, sample s) the replay follows the path the render kernel traces from the stream
(seed, p, sample_offset + s), all paths together, one bounce per round, with the render kernel's own f32 device functions:
the jitter from the documented RNG (restated here in NumPy), Camera::pixel_ray through b200rt_camera_rays continuing the
stream after the two jitter draws, then per bounce b200rt_closest_hit and b200rt_scatter (Material::scatter / ::emitted, or
the sky for a miss), continuing the stream by the draws each bounce took.  What the replay states itself is what the kernel
wires around those functions: the work items' (pixel, sample) keys, ray_color's accumulators, the depth countdown and what
ends a path, the per-sample clamp, the fixed-point sums and the write-back.  Its arithmetic is the kernel's:
`emit + atten * x` is one fmaf (a small g++ helper: rounding the product and sum to float64 first is not always the correctly
rounded f32), `atten * mul` one f32 product, and the pixel is the 2^-32 fixed-point sum converted to f32 once.  No f32 path
is compared with an f64 one, so the accumulation buffer and the rays / paths / depth_exhausted counters must be equal."""
import ctypes as C
import subprocess

import numpy as np
import pytest

from test_scene_update import Arrays, clone

INF = float("inf")
U32 = np.uint32

HELPER_SRC = r"""
#include <cmath>
#include <cstddef>
// a * b + c rounded once, as the device's FFMA
extern "C" void fmaf_n(const float* a, const float* b, const float* c, float* out, size_t n) {
    for (size_t i = 0; i < n; ++i) out[i] = std::fma(a[i], b[i], c[i]);
}
// the kernel's (float) of a 64-bit fixed-point sum: one rounding to nearest
extern "C" void ll_to_f32(const long long* x, float* out, size_t n) {
    for (size_t i = 0; i < n; ++i) out[i] = (float)x[i];
}
"""


@pytest.fixture(scope="module")
def f32ops(tmp_path_factory):
    d = tmp_path_factory.mktemp("replay_helper")
    src, so = d / "helper.cpp", d / "libreplay_helper.so"
    src.write_text(HELPER_SRC)
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-o", str(so), str(src)])
    lib = C.CDLL(str(so))
    lib.fmaf_n.argtypes = [C.c_void_p] * 4 + [C.c_size_t]
    lib.ll_to_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]

    class Ops:
        @staticmethod
        def fmaf(a, b, c):
            a, b, c = (np.ascontiguousarray(x, dtype=np.float32) for x in (a, b, c))
            assert a.shape == b.shape == c.shape
            out = np.empty_like(a)
            lib.fmaf_n(a.ctypes.data, b.ctypes.data, c.ctypes.data, out.ctypes.data, a.size)
            return out

        @staticmethod
        def ll_to_f32(x):
            x = np.ascontiguousarray(x, dtype=np.int64)
            out = np.empty(x.shape, np.float32)
            lib.ll_to_f32(x.ctypes.data, out.ctypes.data, x.size)
            return out
    return Ops


# ---- the RNG of include/b200rt.h (b200rt_rng_uniforms), on uint32 arrays ----------------------------------------------
def _pcg_out(s):
    w = ((s >> ((s >> U32(28)) + U32(4))) ^ s) * U32(277803737)
    return (w >> U32(22)) ^ w


def _hash32(x):
    return _pcg_out(x * U32(747796405) + U32(2891336453))


def uniforms(seed, a, b, n):
    """The first n draws of the streams (seed, a[i], b[i]): float32[n][len(a)], as the device's Rng::gen makes them."""
    a, b = np.atleast_1d(np.asarray(a, U32)), np.atleast_1d(np.asarray(b, U32))
    k0 = _hash32(np.array([seed & 0xFFFFFFFF], U32))
    k1 = _hash32(np.array([seed >> 32], U32) ^ k0)
    state = _hash32(b + _hash32(a ^ k1))
    inc = (_hash32(a + _hash32(b ^ k0)) << U32(1)) | U32(1)
    out = []
    for _ in range(n):
        state = state * U32(747796405) + inc
        out.append((_pcg_out(state) >> U32(8)).astype(np.float32) * np.float32(2.0 ** -24))
    return np.array(out)


def selected_pixels(W, H, rows, shard):
    """Pixel indices (row * W + column) a render of rows [r0, r1) ((0, 0): all) and tile shard (count, index) writes:
    tile t of the 8x4 grid that starts at the row range's first tile row, t % count == index."""
    r0, r1 = rows if tuple(rows) != (0, 0) else (0, H)
    y, x = np.mgrid[r0:r1, 0:W]
    t = (y // 4 - r0 // 4) * ((W + 7) // 8) + x // 8
    keep = t % shard[0] == shard[1]
    return (y[keep] * W + x[keep]).astype(U32)


def replay(rt, ops, scene, cam, seed, samples, max_depth, sample_offset=0, rows=(0, 0), shard=(1, 0), into=None):
    """rt.render's accum[H, W, 4] and (rays, paths, depth_exhausted), and the radiance of every path, from the hooks."""
    H, W = cam.image_height, cam.image_width
    pix = selected_pixels(W, H, rows, shard)
    a = np.repeat(pix, samples)                                    # path i = (pixel a[i], sample b[i])
    b = np.tile(np.arange(samples, dtype=U32), len(pix)) + U32(sample_offset)
    n = len(a)
    u = uniforms(seed, a, b, 2)                                    # draws 0, 1: the jitter
    xy = np.stack([(a % W).astype(np.float32) + u[0], (a // W).astype(np.float32) + u[1]], 1)
    ray, lens = rt.camera_rays(cam, xy, seed, stream=np.stack([a, b, np.full(n, 2, U32)], 1), with_draws=True)
    pos = U32(2) + lens                                            # the first bounce draws after the lens
    alive = np.arange(n)
    atten, emit = np.ones((n, 3), np.float32), np.zeros((n, 3), np.float32)
    radiance = np.zeros((n, 3), np.float32)
    rays = exhausted = 0
    depth = max_depth                                              # every path alive in a round has the same depth left
    while len(alive) and depth > 0:
        ids, hits, _ = rt.closest_hit(scene, ray, 0.001, INF)
        rays += len(alive)
        hits["id"] = ids                                           # -1: a miss, whose record returns the sky
        sc = rt.scatter(scene, ray, hits, seed, stream=np.stack([a[alive], b[alive], pos], 1))
        # a miss: emit + atten * background; a hit: emit + atten * emission (0 unless the material emits), before atten *= mul
        e = ops.fmaf(atten, sc["emitted"], emit)
        end = (ids < 0) | (sc["scattered"] == 0)
        depth -= 1
        if depth == 0:
            exhausted += int((~end).sum())
            end[:] = True
        radiance[alive[end]] = e[end]
        go = ~end
        alive, emit = alive[go], e[go]
        atten = atten[go] * sc["attenuation"][go]
        ray = np.concatenate([sc["o"], sc["d"]], 1)[go]
        pos = pos[go] + sc["draws"][go]

    # acc_add: a sample with a NaN or infinite channel adds nothing; the others are clamped to +-2e9 / samples and
    # summed as 64-bit integers of 2^-32
    lim = np.float32(2.0e9) / np.float32(samples)
    ok = np.isfinite(radiance).all(1)
    v = np.clip(np.where(ok[:, None], radiance, 0), -lim, lim)
    q = np.rint(v.astype(np.float64) * 2.0 ** 32).astype(np.int64)
    sums = q.reshape(len(pix), samples, 3).sum(1)
    rgb = ops.ll_to_f32(sums) * np.float32(2.0 ** -32)
    new = np.concatenate([rgb, np.full((len(pix), 1), samples, np.float32)], 1)
    out = np.zeros((H * W, 4), np.float32) if into is None else into.reshape(H * W, 4).copy()
    out[pix] = new if into is None else new + out[pix]
    return out.reshape(H, W, 4), (rays, n, exhausted), radiance


# ---- the hooks' new arguments -------------------------------------------------------------------------------------------
def test_fmaf_helper_rounds_once(f32ops):
    """1 + 2^-11 + 2^-24 + 2^-77: float64 drops the 2^-77 and lands on a float32 tie, which rounds to even (down);
    the exact value is above the tie, so fmaf rounds up."""
    a, c = np.float32(1 + 2.0 ** -12), np.float32(2.0 ** -77)
    twice = np.float32(np.float64(a) * np.float64(a) + np.float64(c))
    got = f32ops.fmaf(np.array([a]), np.array([a]), np.array([c]))[0]
    assert got == np.float32(1 + 2.0 ** -11 + 2.0 ** -23) and twice == np.float32(1 + 2.0 ** -11)
    big = np.array([2 ** 62 + 2 ** 38 + 1, -(2 ** 40) - 1, 2 ** 24 + 1], np.int64)
    assert list(f32ops.ll_to_f32(big)) == [np.float32(2.0 ** 62 + 2.0 ** 39), np.float32(-(2.0 ** 40)), np.float32(2.0 ** 24)]


def test_numpy_rng_is_the_documented_stream(po):
    for seed, a, b in [(0, 0, 0), (0xDEADBEEF, 123456, 77), (2 ** 63 + 5, 959999, 499)]:
        assert np.array_equal(uniforms(seed, a, b, 64)[:, 0].astype(np.float64), po.rng_uniforms(seed, a, b, 64))


@pytest.mark.gpu
def test_numpy_rng_is_the_device_stream(rt, gpu_required):
    for seed, a, b in [(0, 0, 0), (0xDEADBEEF, 123456, 77), (2 ** 63 + 5, 959999, 499), (9, 2 ** 32 - 1, 2 ** 31 + 3)]:
        assert np.array_equal(uniforms(seed, a, b, 64)[:, 0], rt.rng_uniforms(seed, a, b, 64))


@pytest.mark.gpu
def test_hook_streams_and_miss_records(rt, weekend, gpu_required):
    """stream = (i, 0, 0) is the default stream; a skip of k continues the stream k draws later; the lens draws are counted;
    a miss record returns the sky of its direction and nothing else."""
    rng = np.random.default_rng(4)
    cam = rt.default_camera(120, camera_aperture=0.5)
    n = 4000
    xy = np.stack([rng.uniform(0, 120, n), rng.uniform(0, 80, n)], 1).astype(np.float32)
    idx = np.arange(n, dtype=U32)
    zero = np.zeros(n, U32)
    r0 = rt.camera_rays(cam, xy, 5)
    r1, k = rt.camera_rays(cam, xy, 5, stream=np.stack([idx, zero, zero], 1), with_draws=True)
    assert np.array_equal(r0, r1) and np.all(k >= 2) and np.all(k % 2 == 0) and (k > 2).any()
    # a pair of lens draws inside the unit disk is accepted: with the default stream draws 0, 1 come first, after a skip
    # of 2 draws 2, 3 (margins keep the f32 compare of the device out of the test)
    u = uniforms(5, idx, zero, 4) * np.float32(2) - np.float32(1)
    _, k2 = rt.camera_rays(cam, xy, 5, stream=np.stack([idx, zero, np.full(n, 2, U32)], 1), with_draws=True)
    for draws, r2 in ((k, u[0] ** 2 + u[1] ** 2), (k2, u[2] ** 2 + u[3] ** 2)):
        assert np.all(draws[r2 < 0.999] == 2) and np.all(draws[r2 > 1.001] > 2) and (r2 > 1.001).any()
    lensless = rt.camera((13.0, 2.0, 3.0), (0.0, 0.0, 0.0), vfov=20.0, aperture=None, width=120)
    _, k0 = rt.camera_rays(lensless, xy, 5, stream=np.stack([idx, zero, np.full(n, 7, U32)], 1), with_draws=True)
    assert np.all(k0 == 0)

    ids, hits, _ = rt.closest_hit(weekend, r0, 0.001, INF)
    hits["id"] = ids
    assert (ids >= 0).any() and (ids < 0).any()
    s0 = rt.scatter(weekend, r0, hits, 3)
    s1 = rt.scatter(weekend, r0, hits, 3, stream=np.stack([idx, zero, zero], 1))
    assert np.array_equal(s0, s1)
    miss = ids < 0
    assert np.all(s0["scattered"][miss] == 0) and np.all(s0["draws"][miss] == 0) and np.all(s0["attenuation"][miss] == 0)
    d = r0[miss, 3:].astype(np.float64)
    t = 0.5 * (d[:, 1] / np.linalg.norm(d, axis=1) + 1.0)
    sky = np.stack([1 - t + 0.5 * t, 1 - t + 0.7 * t, np.ones_like(t)], 1)
    np.testing.assert_allclose(s0["emitted"][miss], sky, rtol=0, atol=1e-6)


# ---- the renders ------------------------------------------------------------------------------------------------------
def _lensless(rt, width):
    return rt.camera((13.0, 2.0, 3.0), (0.0, 0.0, 0.0), vfov=20.0, aperture=None, width=width)


def _cornell_cam(rt, width, lens):
    return rt.camera((278, 278, -800), (278, 278, 0), vfov=40, aperture=0.00001 if lens else None, width=width,
                     aspect_ratio=(1, 1), focus_length=10.0)


def _bright_light_scene(rt):
    """A light of 3e9: with 4 samples the clamp (2e9 / 4) takes every sample that sees it."""
    b = rt.SceneBuilder().set_skybox(rt.SkyBox.Flat((0.2, 0.3, 0.4)))
    b.add(rt.Sphere((0.0, -1000.0, 0.0), 1000.0), rt.Lambertian(rt.TextureLoader.solid(0.5, 0.5, 0.5)))
    b.add(rt.Sphere((0.0, 1.0, 0.0), 1.0), rt.DiffuseLight(rt.TextureLoader.solid(3e9, 3e9, 3e9)))
    b.add(rt.Sphere((-2.5, 1.0, 0.5), 1.0), rt.Metal((0.8, 0.8, 0.8), 0.1))
    b.add(rt.Sphere((2.5, 1.0, -0.5), 1.0), rt.Dielectric(1.5))
    return b.finalize()


def _cornell_lit_by_update(rt):
    """Cornell created with its lights turned Lambertian (no emitters), then updated in place to the lit box."""
    dark = clone(rt, rt.Scene.named("cornell", seed=0))
    ad = Arrays(dark)
    lights = np.nonzero((ad.mat_i[:, 0] == rt._ffi.MAT_DIFFUSE_LIGHT) | (ad.mat_i[:, 0] == rt._ffi.MAT_FAIRY_LIGHT))[0]
    kinds = ad.mat_i[lights, 0].copy()
    assert len(lights) > 0
    ad.mat_i[lights, 0] = rt._ffi.MAT_LAMBERTIAN
    dark.device()
    lit = clone(rt, dark)
    Arrays(lit).mat_i[lights, 0] = kinds
    dark.update(lit)
    return dark


# id: scene, camera, width, samples, max_depth, and what else the case selects
CASES = [
    dict(id="random-lens-ragged-d50", scene="random", cam="lens", width=150, spp=4, depth=50),
    dict(id="random-lensless-rows-d5", scene="random", cam="lensless", width=123, spp=4, depth=5, rows=(13, 62)),
    dict(id="random-shard-d1", scene="random", cam="lens", width=120, spp=4, depth=1, shard=(3, 2)),
    dict(id="random-offset-chunks5-d2", scene="random", cam="lens", width=104, spp=8, depth=2, offset=37, env={"B200RT_CHUNKS": "5"}),
    dict(id="random-accumulate-d50", scene="random", cam="lens", width=100, spp=4, depth=50, offset=4, accumulate=True),
    dict(id="random-night-d50", scene="random-night", cam="lens", width=150, spp=6, depth=50),
    dict(id="cornell-lensless-d50", scene="cornell", cam="lensless", width=100, spp=4, depth=50),
    dict(id="cornell-updated-lens-d5", scene="cornell-updated", cam="lens", width=80, spp=4, depth=5),
    dict(id="earth-lens-d50", scene="earth", cam="lens", width=120, spp=4, depth=50),
    dict(id="perlin-exact-slab-d50", scene="perlin", cam="lensless", width=120, spp=4, depth=50, env={"B200RT_FAST_SLAB": "0"}),
    dict(id="scaled-lbvh-d50", scene="scaled", cam="lens", width=100, spp=4, depth=50, env={"B200RT_BUILDER": "lbvh"}),
    dict(id="clamp-lensless-d5", scene="bright", cam="lensless", width=64, spp=4, depth=5),
]


def _scene(rt, name):
    if name == "cornell-updated":
        return _cornell_lit_by_update(rt)
    if name == "bright":
        return _bright_light_scene(rt)
    if name == "scaled":
        return rt.Scene.named("scaled", seed=3, param=40)
    return rt.Scene.named(name, seed=7)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c["id"] for c in CASES])
def test_render_equals_replayed_paths(rt, f32ops, gpu_required, monkeypatch, case):
    for k, v in case.get("env", {}).items():
        monkeypatch.setenv(k, v)
    scene = _scene(rt, case["scene"])
    scene.device()                                                 # created under the case's environment (tree builder)
    W, spp, depth, seed = case["width"], case["spp"], case["depth"], 11
    if case["scene"].startswith("cornell"):
        cam = _cornell_cam(rt, W, case["cam"] == "lens")
    else:
        cam = rt.default_camera(W) if case["cam"] == "lens" else _lensless(rt, W)
    kw = dict(sample_offset=case.get("offset", 0), rows=case.get("rows", (0, 0)), shard=case.get("shard", (1, 0)))
    before = None
    if case.get("accumulate"):
        before, _ = rt.render(scene, cam, samples=3, max_depth=depth, seed=seed + 1)
        assert before[..., :3].sum() > 0
    got, st = rt.render(scene, cam, samples=spp, max_depth=depth, seed=seed, into=None if before is None else before.copy(), **kw)
    want, (rays, paths, exhausted), radiance = replay(rt, f32ops, scene, cam, seed, spp, depth, into=before, **kw)
    bad = np.nonzero((got != want).any(-1))
    assert bad[0].size == 0, (f"{bad[0].size} pixels differ, first (row, column): {list(zip(*bad))[:5]}",
                              got[bad][:3], want[bad][:3])
    assert (st.rays, st.paths, st.depth_exhausted) == (rays, paths, exhausted)
    assert got[..., :3].max() > 0 and (rays == paths if depth == 1 else rays > paths)
    if depth <= 5 and case["scene"] != "bright":
        assert exhausted > 0
    if case["scene"] == "bright":
        assert (radiance > np.float32(2e9) / spp).any()           # some samples were clamped
