"""b200rt_scene_update / Scene.update: a resident scene takes new geometry, materials, textures and image texels in place and
refits its BVH on the device.  Closest hits do not depend on the tree's topology, so after every update the device must give
what the brute-force f32 mirror (oracle/gpu_f32.hpp) gives on the new description, bit for bit, and renders must equal those
of a scene created from it.  An unchanged description must leave every node as the builder emitted it (same traversal
counts), repeated updates must not grow boxes, rejected updates must change nothing, and an update must wait for renders
still in flight on the scene."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_random_scenes import _random_scene, _rays

pytestmark = pytest.mark.gpu
INF = float("inf")
BUILDERS = ("sah", "lbvh")


class Dev:
    """A device handle created from a description; usable wherever the API takes a Scene (it only calls .device())."""

    def __init__(self, rt, desc):
        self.F = rt._ffi
        self.h = C.c_void_p()
        self.F.check(self.F.lib.b200rt_scene_create(desc, -1, C.byref(self.h)))

    def device(self, device=-1):
        return self.h

    def update(self, desc):
        return self.F.lib.b200rt_scene_update(self.h, desc)

    def close(self):
        if self.h:
            self.F.lib.b200rt_scene_destroy(self.h)
            self.h = C.c_void_p()


def _view(ptr, n, width, dtype=np.float32):
    """The n records behind a desc array pointer as an (n, width) array of 4-byte words (a view: writes go to the desc)."""
    if n == 0:
        return np.zeros((0, width), dtype=dtype)
    ct = C.c_float if dtype == np.float32 else C.c_int32
    return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(n, width))


class Arrays:
    """Writable views of a host scene's description: spheres (cx, cy, cz, r), rects (d1_min, d1_max, d2_min, d2_max, offset),
    boxes (min xyz at 0..2, max xyz at 4..6), materials and textures as float and int words."""

    def __init__(self, scene):
        d = scene.desc.contents
        self.d = d
        self.spheres = _view(d.spheres, d.n_spheres, 4)
        self.rects = _view(d.rects, d.n_rects, 8)
        self.boxes = _view(d.boxes, d.n_boxes, 8)
        self.mat_f, self.mat_i = _view(d.materials, d.n_prims, 8), _view(d.materials, d.n_prims, 8, np.int32)
        self.tex_f, self.tex_i = _view(d.textures, d.n_textures, 8), _view(d.textures, d.n_textures, 8, np.int32)

    def copy_from(self, other):
        for a in ("spheres", "rects", "boxes", "mat_i", "tex_i"):
            getattr(self, a)[...] = getattr(other, a)


def clone(rt, scene):
    """A second host scene with the same description (same Perlin seed, so the same tables); its arrays are independent."""
    c = rt.Scene.from_json(scene.to_json())
    Arrays(c).copy_from(Arrays(scene))
    return c


def _hits(rt, dev, rays):
    ids, hits, st = rt.closest_hit(dev, rays, 0.001, INF)
    return ids, hits, (st.node_visits, st.prim_tests)


def _assert_mirror(rt, po, dev, desc, rays, what):
    ids, hits, _ = rt.closest_hit(dev, rays, 0.001, INF)
    want = po.closest_hit_gpu32(desc, rays, 0.001, INF)
    assert np.array_equal(ids, want["id"]), (what, int((ids != want["id"]).sum()))
    hit = ids >= 0
    for f in ("t", "p", "n", "front_face"):
        assert np.array_equal(hits[f][hit], want[f][hit]), (what, f)


def _weekend_cam(rt, width=160):
    return rt.default_camera(width)


# ---- 1. no-op update ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("which", ["weekend", "scaled"])
def test_noop_update_leaves_nodes_unchanged(rt, po, gpu_required, monkeypatch, builder, which):
    """Same description, fresh handle per builder: ids, hit records and traversal counts (so the nodes) are unchanged, for the
    Weekend scene (tree in shared memory) and a 1e5-sphere scene (tree read through L1)."""
    monkeypatch.setenv("B200RT_BUILDER", builder)
    s = rt.Scene.named("random", seed=0xDEADBEEF) if which == "weekend" else rt.Scene.named("scaled", seed=11, param=158)
    dev = Dev(rt, s.desc)
    try:
        inf = rt._ffi.SceneInfo()
        rt._ffi.check(rt._ffi.lib.b200rt_scene_info(dev.h, C.byref(inf)))
        assert (inf.bvh_nodes_in_smem == inf.n_bvh_nodes) == (which == "weekend")
        assert inf.bvh_builder == (1 if builder == "lbvh" else 0)
        scale = 8.0 if which == "weekend" else 158.0
        rays = _rays(np.random.default_rng(5), 30_000, scale)
        ids0, hits0, cnt0 = _hits(rt, dev, rays)
        cam = _weekend_cam(rt, 96) if which == "weekend" else rt.camera((142, 30, 55), (0, 0, 0), vfov=30, width=128, aspect_ratio=(16, 9), focus_length=10.0)
        img0, st0 = rt.render(dev, cam, samples=4, seed=1, count_traversal=True)
        for _ in range(2):
            assert dev.update(s.desc) == 0, rt._ffi.lib.b200rt_last_error()
            ids, hits, cnt = _hits(rt, dev, rays)
            assert np.array_equal(ids, ids0) and hits.tobytes() == hits0.tobytes()
            assert cnt == cnt0, (cnt, cnt0)
            img, st = rt.render(dev, cam, samples=4, seed=1, count_traversal=True)
            assert np.array_equal(img, img0) and st.node_visits == st0.node_visits and st.prim_tests == st0.prim_tests
        rt._ffi.check(rt._ffi.lib.b200rt_scene_info(dev.h, C.byref(inf)))
        assert inf.bvh_builder == (1 if builder == "lbvh" else 0)
    finally:
        dev.close()


# ---- 2. random motion against the f32 mirror --------------------------------------------------------------------------------
def _move(rng, a, spread):
    """Moves and resizes every primitive within its leaf-status class, reassigns materials and retunes textures."""
    n = len(a.spheres)
    if n:
        r = a.spheres[:, 3].copy()
        a.spheres[:, :3] = rng.uniform(-spread, spread, (n, 3))
        new_r = rng.choice([1e-3, 0.2, 1.0, 0.2 * spread], n) * rng.uniform(0.5, 1.5, n)
        a.spheres[:, 3] = np.where(r > 0, new_r, np.where(r < 0, -new_r, 0.0))
    n = len(a.rects)
    if n:
        for lo, hi in ((0, 1), (2, 3)):
            v = np.sort(rng.uniform(-spread, spread, (n, 2)) * rng.choice([0.05, 0.3, 1.0], (n, 1)), axis=1)
            a.rects[:, lo], a.rects[:, hi] = v[:, 0], v[:, 1]
        a.rects[:, 4] = rng.uniform(-spread, spread, n)
    n = len(a.boxes)
    if n:
        lo = rng.uniform(-spread, spread, (n, 3))
        a.boxes[:, 0:3] = lo
        a.boxes[:, 4:7] = lo + rng.choice([1e-5, 0.01, 0.5, 2.0], (n, 3))
    perm = rng.permutation(len(a.mat_i))
    a.mat_i[...] = a.mat_i[perm].copy()
    if len(a.tex_f):
        solid = a.tex_i[:, 0] == 0
        a.tex_f[solid, 1:4] = rng.uniform(0.05, 0.95, (int(solid.sum()), 3))
        a.tex_f[~solid, 4] = rng.uniform(0.5, 6.0, int((~solid).sum()))


@pytest.mark.parametrize("builder", BUILDERS)
@pytest.mark.parametrize("seed", range(4))
def test_random_motion_matches_mirror(rt, po, gpu_required, monkeypatch, builder, seed):
    rng = np.random.default_rng(3000 + seed)
    n = int((17, 300, 2500, 64)[seed])
    spread = float((3.0, 30.0, 2000.0, 30.0)[seed])
    s = _random_scene(rt, rng, n, spread)
    monkeypatch.setenv("B200RT_BUILDER", builder)
    dev = Dev(rt, s.desc)
    try:
        rays = _rays(rng, 40_000, spread)
        _assert_mirror(rt, po, dev, s.desc, rays, "created")
        a = Arrays(s)
        for step in range(4):
            _move(rng, a, spread * (1.0, 0.5, 3.0, 1.0)[step])
            assert dev.update(s.desc) == 0, rt._ffi.lib.b200rt_last_error()
            _assert_mirror(rt, po, dev, s.desc, rays, (seed, builder, step))
    finally:
        dev.close()


def test_primitive_across_the_up_front_threshold(rt, po, gpu_required):
    """A small sphere grown past 30 % of the scene's area stays in the tree, and the ground rect shrunk stays up front:
    only speed depends on the list chosen at creation, hits still match the mirror."""
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    c = clone(rt, s)
    dev = Dev(rt, c.desc)
    try:
        a = Arrays(c)
        small = int(np.argmin(np.where(a.spheres[:, 3] > 0, a.spheres[:, 3], INF)))
        a.spheres[small] = (0.0, 0.0, 0.0, 900.0)
        a.rects[:, 0:4] *= np.float32(0.01)
        assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
        rays = _rays(np.random.default_rng(9), 40_000, 12.0)
        _assert_mirror(rt, po, dev, c.desc, rays, "threshold")
    finally:
        dev.close()


# ---- 3. renders equal a fresh scene's -----------------------------------------------------------------------------------------
def _render_pair(rt, dev, desc, cam, spp=8):
    fresh = Dev(rt, desc)
    try:
        want, sw = rt.render(fresh, cam, samples=spp, seed=4, count_traversal=True)
    finally:
        fresh.close()
    got, sg = rt.render(dev, cam, samples=spp, seed=4, count_traversal=True)
    return got, want, sg, sw


def test_render_after_update_equals_fresh_weekend(rt, gpu_required):
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    c = clone(rt, s)
    dev = Dev(rt, c.desc)
    try:
        a = Arrays(c)
        small = (a.spheres[:, 3] > 0) & (a.spheres[:, 3] < 0.5)
        rng = np.random.default_rng(1)
        a.spheres[small, 0] += rng.uniform(-0.4, 0.4, int(small.sum()))
        a.spheres[small, 2] += rng.uniform(-0.4, 0.4, int(small.sum()))
        a.spheres[small, 1] += rng.uniform(0.0, 0.6, int(small.sum()))
        assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
        got, want, _, _ = _render_pair(rt, dev, c.desc, _weekend_cam(rt))
        assert np.array_equal(got, want)
        before, _ = rt.render(s, _weekend_cam(rt), samples=8, seed=4)
        assert not np.array_equal(got, before)     # the motion is visible
    finally:
        dev.close()


def test_render_after_update_equals_fresh_cornell_emitter_flip(rt, gpu_required):
    """A Lambertian turned into a DiffuseLight flips has_emitters on: the scene starts from Cornell with its ceiling light
    turned Lambertian, so it has no emitter at creation."""
    s = rt.Scene.named("cornell", seed=0)
    cam = rt.camera((278, 278, -800), (278, 278, 0), vfov=40, aperture=None, width=80, aspect_ratio=(1, 1), focus_length=10.0)
    dark = clone(rt, s)
    ad = Arrays(dark)
    lights = np.nonzero((ad.mat_i[:, 0] == 3) | (ad.mat_i[:, 0] == 4))[0]
    assert len(lights) > 0
    ad.mat_i[lights, 0] = 2
    dev = Dev(rt, dark.desc)
    try:
        c = clone(rt, dark)
        a = Arrays(c)
        lamb = np.nonzero(a.mat_i[:, 0] == 2)[0]
        a.mat_i[lamb[0], 0] = 3
        assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
        got, want, _, _ = _render_pair(rt, dev, c.desc, cam, spp=16)
        assert np.array_equal(got, want) and got[..., :3].max() > 0
    finally:
        dev.close()


def test_render_after_update_equals_fresh_earth_texels(rt, gpu_required):
    s = rt.Scene.named("earth")
    c = clone(rt, s)
    dev = Dev(rt, c.desc)
    try:
        img = c.desc.contents.images[0]
        w, h = img.width, img.height
        texels = np.ctypeslib.as_array(img.rgb8, shape=(h * w * 3,)).copy()
        texels = (255 - texels).astype(np.uint8)          # a new picture of the same size, owned here
        img.rgb8 = texels.ctypes.data_as(C.POINTER(C.c_uint8))
        assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
        cam = rt.camera((13, 2, 3), (0, 0, 0), vfov=20, aperture=None, width=96, aspect_ratio=(16, 9), focus_length=10.0)
        got, want, _, _ = _render_pair(rt, dev, c.desc, cam)
        assert np.array_equal(got, want)
        old, _ = rt.render(s, cam, samples=8, seed=4)
        assert not np.array_equal(got, old)
    finally:
        dev.close()


# ---- 4. drift ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("builder", BUILDERS)
def test_hundred_updates_then_back_equals_original(rt, gpu_required, monkeypatch, builder):
    monkeypatch.setenv("B200RT_BUILDER", builder)
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    orig = Arrays(s)
    base = orig.spheres.copy()
    c = clone(rt, s)
    a = Arrays(c)
    dev = Dev(rt, c.desc)
    cam = _weekend_cam(rt, 96)
    rays = _rays(np.random.default_rng(2), 20_000, 8.0)
    try:
        img0, st0 = rt.render(dev, cam, samples=4, seed=7, count_traversal=True)
        ids0, hits0, cnt0 = _hits(rt, dev, rays)
        small = (base[:, 3] > 0) & (base[:, 3] < 0.5)
        phase = np.random.default_rng(3).uniform(0, 2 * np.pi, len(base))
        for k in range(100):
            a.spheres[small, 1] = base[small, 1] + 1.5 * np.abs(np.sin(0.2 * k + phase[small]))
            assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
        a.copy_from(orig)
        assert dev.update(c.desc) == 0
        img, st = rt.render(dev, cam, samples=4, seed=7, count_traversal=True)
        ids, hits, cnt = _hits(rt, dev, rays)
        assert np.array_equal(img, img0) and (st.node_visits, st.prim_tests) == (st0.node_visits, st0.prim_tests)
        assert np.array_equal(ids, ids0) and hits.tobytes() == hits0.tobytes() and cnt == cnt0
    finally:
        dev.close()


# ---- 5. fast-slab guard ---------------------------------------------------------------------------------------------------------
def test_scale_up_and_back_follows_the_slab_guard(rt, po, gpu_required):
    """Scaled by 1e4 the padding and the origin bound of the fast slab test grow with the scene; rays from origins far
    outside the unscaled scene are then on the fast path, and must still find every hit."""
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    c = clone(rt, s)
    a = Arrays(c)
    orig = Arrays(s)
    dev = Dev(rt, c.desc)
    try:
        for scale in (1e4, 1.0):
            a.copy_from(orig)
            a.spheres[...] *= np.float32(scale)
            a.boxes[:, [0, 1, 2, 4, 5, 6]] *= np.float32(scale)
            a.rects[:, :5] *= np.float32(scale)
            assert dev.update(c.desc) == 0, rt._ffi.lib.b200rt_last_error()
            rays = _rays(np.random.default_rng(4), 30_000, 8.0 * scale)
            _assert_mirror(rt, po, dev, c.desc, rays, scale)
            fresh = Dev(rt, c.desc)
            try:
                ids_f, hits_f, _ = rt.closest_hit(fresh, rays, 0.001, INF)
                cam = rt.camera((13 * scale, 2 * scale, 3 * scale), (0, 0, 0), vfov=20, aperture=0.1 * scale, width=96, aspect_ratio=(3, 2), focus_length=10.0 * scale)
                want, _ = rt.render(fresh, cam, samples=4, seed=5)
            finally:
                fresh.close()
            ids, hits, _ = rt.closest_hit(dev, rays, 0.001, INF)
            assert np.array_equal(ids, ids_f) and hits.tobytes() == hits_f.tobytes()
            got, _ = rt.render(dev, cam, samples=4, seed=5)
            assert np.array_equal(got, want), scale
    finally:
        dev.close()


# ---- 6. rejections --------------------------------------------------------------------------------------------------------------
def _reject_cases(rt):
    def n_prims(c):
        c.desc.contents.n_prims -= 1

    def prim_index(c):
        d = c.desc.contents
        sph = [i for i in range(d.n_prims) if d.prims[i].type == 0]
        d.prims[sph[0]].index, d.prims[sph[1]].index = d.prims[sph[1]].index, d.prims[sph[0]].index

    def prim_type(c):
        d = c.desc.contents
        i = [k for k in range(d.n_prims) if d.prims[k].type == 0][0]
        d.prims[i].type, d.prims[i].index = 4, 0   # a box record exists (Weekend's coat box)

    def count(c):
        c.desc.contents.n_spheres += 1

    def radius(c):
        a = Arrays(c)
        a.spheres[5, 3] = -a.spheres[5, 3]

    def nan(c):
        Arrays(c).spheres[7, 0] = np.nan

    return {"n_prims": n_prims, "prim_index": prim_index, "prim_type": prim_type, "count": count, "radius": radius, "nan": nan}


@pytest.mark.parametrize("case", ["n_prims", "prim_index", "prim_type", "count", "radius", "nan", "image_size"])
def test_rejected_update_changes_nothing(rt, gpu_required, case):
    F = rt._ffi
    s = rt.Scene.named("earth" if case == "image_size" else "random", seed=0xDEADBEEF)
    dev = Dev(rt, s.desc)
    cam = _weekend_cam(rt, 96)
    rays = _rays(np.random.default_rng(6), 20_000, 8.0)
    try:
        ids0, hits0, cnt0 = _hits(rt, dev, rays)
        img0, _ = rt.render(dev, cam, samples=4, seed=2)
        c = clone(rt, s)
        Arrays(c).spheres[:, 1] += 0.25                 # a valid motion riding along, which must not be applied either
        if case == "image_size":
            c.desc.contents.images[0].width -= 1
        else:
            _reject_cases(rt)[case](c)
        assert dev.update(c.desc) == F.EINVAL
        assert F.lib.b200rt_last_error()
        ids, hits, cnt = _hits(rt, dev, rays)
        assert np.array_equal(ids, ids0) and hits.tobytes() == hits0.tobytes() and cnt == cnt0
        img, _ = rt.render(dev, cam, samples=4, seed=2)
        assert np.array_equal(img, img0)
    finally:
        dev.close()


# ---- 7. ordering --------------------------------------------------------------------------------------------------------------
def test_update_waits_for_a_render_in_flight(rt, gpu_required):
    import torch
    F = rt._ffi
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    c = clone(rt, s)
    dev = Dev(rt, c.desc)
    cam = _weekend_cam(rt, 640)
    try:
        want, _ = rt.render(dev, cam, samples=512, seed=8)
        acc = torch.zeros((cam.image_height, cam.image_width, 4), dtype=torch.float32, device="cuda")
        stream = torch.cuda.Stream()
        p = F.RenderParams(samples=512, max_depth=50, seed=8, device=-1)
        a = Arrays(c)
        a.spheres[:, 1] += 0.3
        a.mat_i[...] = a.mat_i[np.random.default_rng(0).permutation(len(a.mat_i))].copy()
        F.check(F.lib.b200rt_render_device(dev.h, C.byref(cam), C.byref(p), C.c_void_p(acc.data_ptr()), C.c_void_p(stream.cuda_stream)))
        assert dev.update(c.desc) == 0, F.lib.b200rt_last_error()
        F.check(F.lib.b200rt_render_device_finish(dev.h, C.c_void_p(stream.cuda_stream), None))
        torch.cuda.synchronize()
        assert np.array_equal(acc.cpu().numpy(), want)
        after, _ = rt.render(dev, cam, samples=4, seed=8)
        fresh = Dev(rt, c.desc)
        try:
            assert np.array_equal(after, rt.render(fresh, cam, samples=4, seed=8)[0])
        finally:
            fresh.close()
    finally:
        dev.close()


# ---- Python face --------------------------------------------------------------------------------------------------------------
def test_scene_update_python(rt, po, gpu_required):
    """Scene.update: the device copy takes the new description, `desc` follows it, and a rejected update raises and leaves
    both the device copy and the host arrays as they were."""
    s = rt.Scene.named("random", seed=0xDEADBEEF)
    s.device()
    rays = _rays(np.random.default_rng(8), 20_000, 8.0)
    nxt = clone(rt, s)
    Arrays(nxt).spheres[:, 1] += 0.5
    want_y = Arrays(nxt).spheres[:, 1].copy()
    s.update(nxt)
    assert np.array_equal(Arrays(s).spheres[:, 1], want_y) and not nxt._host
    _assert_mirror(rt, po, s, s.desc, rays, "python")
    ids0, _, _ = rt.closest_hit(s, rays)
    bad = clone(rt, s)
    bad.desc.contents.n_prims -= 1
    with pytest.raises(rt._ffi.B200rtError):
        s.update(bad)
    assert s.desc.contents.n_prims == bad.desc.contents.n_prims + 1
    assert np.array_equal(rt.closest_hit(s, rays)[0], ids0)
