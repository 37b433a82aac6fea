"""Python face of the host mirror: the reference's builder API, names and argument meaning
(``raytracer`` crate: scene/mod.rs, geometry/, material/, camera/mod.rs; ``src/scenes.rs``).

Nothing here computes: builders serialise to the reference's serde JSON wire format
(src/scenes.rs:128-134,140-143) and hand it to the C++ host (host/raytracer.hpp), which
flattens it and calls the CUDA library through include/b200rt.h.
"""
from __future__ import annotations

import ctypes as C
import json
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import _ffi as F

lib = F.lib


# ---- core ------------------------------------------------------------------------------------
def _vec(v: Sequence[float]) -> dict:
    x, y, z = (float(c) for c in v)
    return {"vec": [x, y, z]}   # nalgebra Vector3 serde form (core/vec3.rs:29-32)


# ---- geometry (geometry/sphere.rs, geometry/rect.rs) --------------------------------------
@dataclass
class Sphere:
    center: Sequence[float]
    radius: float

    def to_json(self):
        return {"Sphere": {"center": _vec(self.center), "radius": float(self.radius)}}


@dataclass
class _Rect:
    tag: str
    d1_min: float
    d1_max: float
    d2_min: float
    d2_max: float
    offset: float

    def to_json(self):
        return {self.tag: {"d1_min": float(self.d1_min), "d1_max": float(self.d1_max), "d2_min": float(self.d2_min),
                           "d2_max": float(self.d2_max), "offset": float(self.offset)}}


def xy_rect(d1_min, d1_max, d2_min, d2_max, offset):   # rect.rs:15
    return _Rect("RectXY", d1_min, d1_max, d2_min, d2_max, offset)


def yz_rect(d1_min, d1_max, d2_min, d2_max, offset):   # rect.rs:25
    return _Rect("RectYZ", d1_min, d1_max, d2_min, d2_max, offset)


def xz_rect(d1_min, d1_max, d2_min, d2_max, offset):   # rect.rs:35
    return _Rect("RectXZ", d1_min, d1_max, d2_min, d2_max, offset)


@dataclass
class RectBox:   # RectBox::new(p0, p1), rect.rs:112
    p0: Sequence[float]
    p1: Sequence[float]

    def to_json(self):
        p0, p1 = [float(c) for c in self.p0], [float(c) for c in self.p1]
        side = lambda a, b, c, d, k: {"d1_min": a, "d1_max": b, "d2_min": c, "d2_max": d, "offset": k}
        return {"RectBox": {
            "min": _vec(p0), "max": _vec(p1),
            "xy_sides": [side(p0[0], p1[0], p0[1], p1[1], p1[2]), side(p0[0], p1[0], p0[1], p1[1], p0[2])],
            "yz_sides": [side(p0[1], p1[1], p0[2], p1[2], p1[0]), side(p0[1], p1[1], p0[2], p1[2], p0[0])],
            "xz_sides": [side(p0[0], p1[0], p0[2], p1[2], p1[1]), side(p0[0], p1[0], p0[2], p1[2], p0[1])]}}


# ---- textures (material/texture/loader.rs:17-46) ------------------------------------------
class TextureLoader:
    def __init__(self, js):
        self.js = js

    @staticmethod
    def solid(r, g, b):
        return TextureLoader({"Solid": _vec((r, g, b))})

    @staticmethod
    def solid_from_vec(v):
        return TextureLoader({"Solid": _vec(v)})

    @staticmethod
    def checker(size, odd: "TextureLoader", even: "TextureLoader"):
        return TextureLoader({"Checker": {"size": float(size), "odd": odd.js, "even": even.js}})

    @staticmethod
    def noise(scalar):
        return TextureLoader({"Perlin": float(scalar)})

    EarthBuiltin: "TextureLoader"

    @staticmethod
    def ImagePath(path: str):
        return TextureLoader({"ImagePath": str(path)})

    def to_json(self):
        return self.js


TextureLoader.EarthBuiltin = TextureLoader("EarthBuiltin")


# ---- materials (material/*.rs) ---------------------------------------------------------------
class Lambertian:
    def __init__(self, texture: TextureLoader):   # Lambertian::new, lambertian.rs:16
        self.albedo = texture

    def to_json(self):
        return {"Lambertian": {"albedo": self.albedo.to_json()}}


class DiffuseLight:
    def __init__(self, texture: TextureLoader):   # lighting.rs:16
        self.albedo = texture

    def to_json(self):
        return {"DiffuseLight": {"albedo": self.albedo.to_json()}}


class FairyLight:
    def __init__(self, texture: TextureLoader):   # lighting.rs:37
        self.albedo = texture

    def to_json(self):
        return {"FairyLight": {"albedo": self.albedo.to_json()}}


class Metal:
    def __init__(self, albedo: Sequence[float], fuzz: Optional[float] = None):   # Metal::new, metal.rs:17-23
        f = 0.0 if fuzz is None else float(fuzz)
        self.albedo, self.fuzz = albedo, min(f, 1.0) if f > 1.0 else f

    def to_json(self):
        return {"Metal": {"albedo": _vec(self.albedo), "fuzz": float(self.fuzz)}}


@dataclass
class Dielectric:   # dielectric.rs:10-13
    ir: float

    def to_json(self):
        return {"Dielectric": {"ir": float(self.ir)}}


# ---- skybox (skybox/mod.rs:11-16) -------------------------------------------------------------
class SkyBox:
    def __init__(self, js):
        self.js = js

    Above: "SkyBox"
    None_: "SkyBox"

    @staticmethod
    def Flat(color):
        return SkyBox({"Flat": _vec(color)})


SkyBox.Above = SkyBox("Above")
SkyBox.None_ = SkyBox("None")


# ---- scene (scene/mod.rs:79-138) -----------------------------------------------------------------
class Scene:
    """A finalized scene: the C++ host's flattened arrays plus (lazily) the device copy."""

    def __init__(self, host_handle: int):
        self._host = C.c_void_p(host_handle)
        self._dev = {}

    @property
    def desc(self) -> "C.POINTER(F.SceneDesc)":
        return lib.b200rt_host_scene_desc(self._host)

    def device(self, device: int = -1) -> C.c_void_p:
        if device not in self._dev:
            h = C.c_void_p()
            F.check(lib.b200rt_scene_create(self.desc, device, C.byref(h)))
            self._dev[device] = h
        return self._dev[device]

    def info(self, device: int = -1) -> F.SceneInfo:
        out = F.SceneInfo()
        F.check(lib.b200rt_scene_info(self.device(device), C.byref(out)))
        return out

    def update(self, new: "Scene") -> None:
        """Take `new`'s contents in place (b200rt_scene_update on every device copy): geometry, materials, textures, image
        texels, Perlin tables and skybox may change, while the primitive list (types and indices), the array counts, the image
        sizes and whether each primitive's box is valid (e.g. a sphere's radius may not cross zero) must stay as they were.
        Each device copy keeps its BVH topology and refits its boxes on the device, so hits and renders equal those of a scene
        created from `new`, bit for bit; only the tree's quality can drift. A rejected update raises B200rtError and changes
        nothing. On success `new`'s host arrays become this scene's own (so `desc`, `to_json` and later `device()` calls see
        them) and `new` is closed. With no device copy yet, the scene simply takes `new`'s contents."""
        if new is self:
            raise ValueError("a scene cannot be updated from itself")
        for h in self._dev.values():
            F.check(lib.b200rt_scene_update(h, new.desc))
        self._host, new._host = new._host, self._host
        new.close()

    def to_json(self) -> str:
        p, n = C.c_void_p(), C.c_size_t()
        F.check(lib.b200rt_host_scene_to_json(self._host, C.byref(p), C.byref(n)), host=True)
        try:
            return C.string_at(p, n.value).decode()
        finally:
            lib.b200rt_free(p)

    def close(self):
        for h in self._dev.values():
            lib.b200rt_scene_destroy(h)
        self._dev = {}
        if self._host:
            lib.b200rt_host_scene_destroy(self._host)
            self._host = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def named(name: str, seed: int = 0xDEADBEEF, param: int = 0) -> "Scene":
        """Scene factories of src/scenes.rs (random, random-night, earth, perlin, box-light,
        cornell, demo) plus the synthetic `scaled` / `lattice` workloads."""
        h = C.c_void_p()
        F.check(lib.b200rt_host_scene_named(name.encode(), seed, param, C.byref(h)), host=True)
        return Scene(h.value)

    @staticmethod
    def from_json(text: str, perlin_seed: int = 0x5EED) -> "Scene":
        h = C.c_void_p()
        b = text.encode()
        F.check(lib.b200rt_host_scene_from_json(b, len(b), perlin_seed, C.byref(h)), host=True)
        return Scene(h.value)


class SceneBuilder:
    def __init__(self):   # Default: skybox Above, scene/mod.rs:85-92
        self.skybox = SkyBox.Above
        self.objects = []

    def set_skybox(self, skybox: SkyBox) -> "SceneBuilder":
        self.skybox = skybox
        return self

    def add(self, geometry, material) -> None:   # scene/mod.rs:98-109
        self.objects.append((geometry, material))

    def to_json(self) -> str:
        return json.dumps({"skybox": self.skybox.js,
                           "objects": [{"geometry": g.to_json(), "material": m.to_json()} for g, m in self.objects]})

    def finalize(self, perlin_seed: int = 0x5EED) -> Scene:   # scene/mod.rs:111-137
        return Scene.from_json(self.to_json(), perlin_seed)


def register_image(name: str, rgb: np.ndarray) -> None:
    """Decoded RGB8 pixels for TextureLoader.EarthBuiltin (name "EarthBuiltin") / ImagePath(name)."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    h, w, c = rgb.shape
    assert c == 3
    F.check(lib.b200rt_host_register_image(name.encode(), w, h, rgb.ctypes.data), host=True)


def decode_image(data: bytes) -> np.ndarray:
    """image::load_from_memory (image_texture.rs:18-21) for a JPEG or PNG: (H, W, 3) uint8, alpha dropped."""
    buf = (C.c_uint8 * len(data)).from_buffer_copy(data)
    w, h, out = C.c_uint32(), C.c_uint32(), C.c_void_p()
    F.check(lib.b200rt_host_decode_image(buf, len(data), C.byref(w), C.byref(h), C.byref(out)), host=True)
    try:
        return np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(h.value, w.value, 3)).copy()
    finally:
        lib.b200rt_free(out)


def checkpoint_save(path: str, accum: np.ndarray, samples_done: int, seed: int) -> None:
    """Write an accumulation-buffer checkpoint ((H, W, 4) float32 sums + the state to continue the sample sequence)."""
    accum = np.ascontiguousarray(accum, dtype=np.float32)
    h, w, c = accum.shape
    assert c == 4
    F.check(lib.b200rt_host_checkpoint_save(str(path).encode(), accum.ctypes.data, w, h, samples_done, seed), host=True)


def checkpoint_load(path: str):
    """-> (accum (H, W, 4) float32, samples_done, seed)"""
    w, h, n, seed, out = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint64(), C.c_void_p()
    F.check(lib.b200rt_host_checkpoint_load(str(path).encode(), C.byref(w), C.byref(h), C.byref(n), C.byref(seed), C.byref(out)), host=True)
    try:
        acc = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_float)), shape=(h.value, w.value, 4)).copy()
    finally:
        lib.b200rt_free(out)
    return acc, n.value, seed.value


decode_jpeg = decode_image


# ---- camera (camera/mod.rs) -------------------------------------------------------------------------
def camera(look_from, look_at, up=(0.0, 1.0, 0.0), *, vfov=20.0, focal_length=1.0, aperture: Optional[float] = 0.001,
           width: int = 0, height: int = 0, aspect_ratio=(3, 2), focus_length: float = 0.0) -> F.Camera:
    """CameraBuilder{vfov,aperture,focal_length,aspect_ratio,width}.build() + CameraPosition::look_at."""
    out = F.Camera()
    d3 = C.c_double * 3
    rn, rd = aspect_ratio if aspect_ratio else (0, 0)
    F.check(lib.b200rt_host_camera(d3(*look_from), d3(*look_at), d3(*up), vfov, focal_length,
                                   -1.0 if aperture is None else aperture, width, height, rn, rd, focus_length,
                                   C.byref(out)), host=True)
    return out


def default_camera(width=640, camera_fov=20.0, camera_focal_length=1.0, camera_aperture=0.001, aspect_ratio=(3, 2)) -> F.Camera:
    """src/scenes.rs:214-231 with the CLI defaults of src/argparse.rs:3-10."""
    out = F.Camera()
    F.check(lib.b200rt_host_default_camera(width, camera_fov, camera_focal_length, camera_aperture, aspect_ratio[0],
                                           aspect_ratio[1], C.byref(out)), host=True)
    return out


# ---- render (src/main.rs:65-130, render.rs) ------------------------------------------------------------
def render(scene: Scene, cam: F.Camera, samples: int = 100, max_depth: int = 50, seed: int = 0, *, sample_offset: int = 0,
           rows=(0, 0), shard=(1, 0), count_traversal: bool = False, device: int = -1, into: Optional[np.ndarray] = None):
    """The frame loop of render_scene: returns (accum[H, W, 4] float32 {sum r,g,b, n}, Stats).
    Row 0 is the bottom of the picture (image.rs:36-38).  `into` = an earlier result (or a checkpoint):
    the new samples are ADDED to it (progressive rendering; give sample_offset = samples already done)."""
    H, W = cam.image_height, cam.image_width
    flags = F.FLAG_COUNT_TRAVERSAL if count_traversal else 0
    if into is not None:
        if into.shape != (H, W, 4) or into.dtype != np.float32 or not into.flags.c_contiguous:
            raise ValueError("`into` must be a C-contiguous float32 array of shape (H, W, 4)")
        accum, flags = into, flags | F.FLAG_ACCUMULATE
    else:
        accum = np.empty((H, W, 4), dtype=np.float32)
    p = F.RenderParams(samples=samples, sample_offset=sample_offset, max_depth=max_depth,
                       flags=flags, seed=seed, row_begin=rows[0], row_end=rows[1],
                       shard_count=shard[0], shard_index=shard[1], device=-1)
    st = F.Stats()
    F.check(lib.b200rt_render(scene.device(device), C.byref(cam), C.byref(p), accum.ctypes.data, C.byref(st)))
    return accum, st


def render_adaptive(scene: Scene, cam: F.Camera, max_samples: int, threshold: float, initial_samples: int = 16, max_depth: int = 50,
                    seed: int = 0, *, sample_offset: int = 0, rows=(0, 0), count_traversal: bool = False, device: int = -1):
    """Tile-adaptive sampling (b200rt_render_adaptive): every 8x4 tile is rendered in passes of doubling sample counts,
    from `initial_samples` up to at most `max_samples`, until its estimated standard error after to_image's gamma is at most
    `threshold` (0..1 output units; 1/255 is about one 8-bit level).  Returns (accum[H, W, 4] float32 {sum r,g,b, n} with
    n the pixel's own sample count, tile_error[ceil(H/4), ceil(W/8)] float32 (each tile's last estimate, -1 outside `rows`;
    row 0 is the bottom, as in accum), Stats)."""
    H, W = cam.image_height, cam.image_width
    accum = np.empty((H, W, 4), dtype=np.float32)
    tile_error = np.empty(((H + 3) // 4, (W + 7) // 8), dtype=np.float32)
    p = F.RenderParams(sample_offset=sample_offset, max_depth=max_depth, flags=F.FLAG_COUNT_TRAVERSAL if count_traversal else 0,
                       seed=seed, row_begin=rows[0], row_end=rows[1], device=-1)
    ad = F.AdaptiveParams(initial_samples=initial_samples, max_samples=max_samples, threshold=threshold)
    st = F.Stats()
    F.check(lib.b200rt_render_adaptive(scene.device(device), C.byref(cam), C.byref(p), C.byref(ad), accum.ctypes.data, None,
                                       tile_error.ctypes.data, C.byref(st)))
    return accum, tile_error, st


def render_denoised(scene: Scene, cam: F.Camera, samples: int, feature_samples: int = 4, iterations: int = 5, max_depth: int = 50,
                    seed: int = 0, *, sample_offset: int = 0, count_traversal: bool = False, device: int = -1):
    """A `samples`-spp frame reconstructed by the feature-guided à-trous filter (b200rt_render_denoised).  Returns
    (denoised[H, W, 4] float32 {mean * n, n}, accum[H, W, 4] float32 (the plain `samples`-spp render, bit for bit),
    features[2, H, W, 4] float32 (plane 0: mean normal xyz and hit distance, plane 1: mean albedo and 0), Stats).
    resolve_rgb8(denoised, samples=0) gives the picture."""
    H, W = cam.image_height, cam.image_width
    denoised = np.empty((H, W, 4), dtype=np.float32)
    accum = np.empty((H, W, 4), dtype=np.float32)
    features = np.empty((2, H, W, 4), dtype=np.float32)
    p = F.RenderParams(samples=samples, sample_offset=sample_offset, max_depth=max_depth,
                       flags=F.FLAG_COUNT_TRAVERSAL if count_traversal else 0, seed=seed, device=-1)
    dn = F.DenoiseParams(feature_samples=feature_samples, iterations=iterations)
    st = F.Stats()
    F.check(lib.b200rt_render_denoised(scene.device(device), C.byref(cam), C.byref(p), C.byref(dn), accum.ctypes.data,
                                       denoised.ctypes.data, features.ctypes.data, None, C.byref(st)))
    return denoised, accum, features, st


def denoise(accum_a: np.ndarray, accum_b: np.ndarray, features: np.ndarray, iterations: int = 5, device: int = -1) -> np.ndarray:
    """The filter of render_denoised alone (b200rt_denoise): two independent accumulation buffers of the same pixels
    ([H, W, 4] {sum r,g,b, count}) and their features ([2, H, W, 4]) -> [H, W, 4] float32 {mean * n, n}."""
    a = np.ascontiguousarray(accum_a, dtype=np.float32)
    b = np.ascontiguousarray(accum_b, dtype=np.float32)
    f = np.ascontiguousarray(features, dtype=np.float32)
    H, W = a.shape[:2]
    if a.shape != (H, W, 4) or b.shape != (H, W, 4) or f.shape != (2, H, W, 4):
        raise ValueError("accum_a and accum_b must be (H, W, 4) and features (2, H, W, 4)")
    out = np.empty((H, W, 4), dtype=np.float32)
    F.check(lib.b200rt_denoise(a.ctypes.data, b.ctypes.data, f.ctypes.data, W, H, iterations, out.ctypes.data, device))
    return out


def resolve_rgb8(accum: np.ndarray, samples: int = 0, device: int = -1) -> np.ndarray:
    """to_image's pixel loop (image.rs:34-40): mean, sqrt gamma, saturating u8, vertical flip."""
    accum = np.ascontiguousarray(accum, dtype=np.float32)
    H, W, _ = accum.shape
    out = np.empty((H, W, 3), dtype=np.uint8)
    F.check(lib.b200rt_resolve_rgb8(accum.ctypes.data, W, H, samples, out.ctypes.data, device))
    return out


def write_png(path: str, rgb8: np.ndarray) -> None:
    rgb8 = np.ascontiguousarray(rgb8, dtype=np.uint8)
    H, W, _ = rgb8.shape
    F.check(lib.b200rt_write_png(str(path).encode(), rgb8.ctypes.data, W, H))


def render_scene(scene: Scene, cam: F.Camera, samples: int = 100, max_reflect: int = 50, output: Optional[str] = "out.png",
                 seed: int = 0, device: int = -1):
    """render_scene(args, scene, camera, pos) (src/main.rs:65-130): returns (rgb8[H, W, 3], Stats)."""
    H, W = cam.image_height, cam.image_width
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    st = F.Stats()
    F.check(lib.b200rt_host_render_scene(scene._host, C.byref(cam), samples, max_reflect, seed, device,
                                         None if output is None else str(output).encode(), rgb.ctypes.data, C.byref(st)), host=True)
    return rgb, st


def render_scene_multi(scene: Scene, cam: F.Camera, samples: int = 100, max_reflect: int = 50, devices: Sequence[int] = (0,),
                       output: Optional[str] = None, seed: int = 0):
    """render_scene on several GPUs from this one process (b200rt_render_rgb8_multi): `samples` is the total per pixel,
    split into sample ranges over `devices`; returns (rgb8[H, W, 3], Stats)."""
    H, W = cam.image_height, cam.image_width
    rgb = np.empty((H, W, 3), dtype=np.uint8)
    devs = (C.c_int * len(devices))(*devices)
    p = F.RenderParams(samples=samples, max_depth=max_reflect, seed=seed, device=-1)
    st = F.Stats()
    F.check(lib.b200rt_render_rgb8_multi(scene.desc, devs, len(devices), C.byref(cam), C.byref(p), rgb.ctypes.data, C.byref(st)))
    if output:
        write_png(output, rgb)
    return rgb, st


# ---- parity hooks ------------------------------------------------------------------------------------------
def as_rays(rays) -> np.ndarray:
    r = np.ascontiguousarray(rays, dtype=np.float32)
    assert r.ndim == 2 and r.shape[1] == 6
    return r


HIT_DTYPE = np.dtype([("t", "<f4"), ("p", "<f4", 3), ("n", "<f4", 3), ("u", "<f4"), ("v", "<f4"), ("front_face", "<i4"), ("id", "<i4")])
SCATTER_DTYPE = np.dtype([("o", "<f4", 3), ("d", "<f4", 3), ("attenuation", "<f4", 3), ("emitted", "<f4", 3), ("scattered", "<i4"), ("draws", "<u4")])
assert HIT_DTYPE.itemsize == C.sizeof(F.Hit) and SCATTER_DTYPE.itemsize == C.sizeof(F.Scatter)


def closest_hit(scene: Scene, rays, t_min: float = 0.001, t_max: float = float("inf"), want_hits: bool = True, device: int = -1):
    """Scene::hit over a ray array (bvh/bbox_tree.rs:56-91): (ids int32[n], hits HIT_DTYPE[n] | None, Stats)."""
    r = as_rays(rays)
    n = r.shape[0]
    ids = np.empty(n, dtype=np.int32)
    hits = np.zeros(n, dtype=HIT_DTYPE) if want_hits else None
    st = F.Stats()
    F.check(lib.b200rt_closest_hit(scene.device(device), r.ctypes.data, n, t_min, t_max, ids.ctypes.data,
                                   hits.ctypes.data if want_hits else None, C.byref(st)))
    return ids, hits, st


def aabb_hit(boxes6, rays, t_min=0.0, t_max=float("inf"), device: int = -1) -> np.ndarray:
    b = np.ascontiguousarray(boxes6, dtype=np.float32)
    r = as_rays(rays)
    out = np.empty(r.shape[0], dtype=np.uint8)
    F.check(lib.b200rt_aabb_hit(b.ctypes.data, r.ctypes.data, r.shape[0], t_min, t_max, out.ctypes.data, device))
    return out.astype(bool)


def _as_stream(stream, n: int):
    """None, or (n, 3) uint32 stream positions (a, b, skip): record i draws from stream (seed, a, b) after `skip` draws."""
    if stream is None:
        return None
    s = np.ascontiguousarray(stream, dtype=np.uint32)
    if s.shape != (n, 3):
        raise ValueError(f"stream must have shape ({n}, 3)")
    return s


def scatter(scene: Scene, rays, hits: np.ndarray, seed: int = 0, device: int = -1, *, stream=None) -> np.ndarray:
    """Material::scatter + ::emitted per record (b200rt_scatter); a record with id -1 is a miss and returns the
    background of its direction as `emitted`.  `stream`: see _as_stream (None: record i draws from (seed, i, 0))."""
    r = as_rays(rays)
    h = np.ascontiguousarray(hits, dtype=HIT_DTYPE)
    s = _as_stream(stream, r.shape[0])
    out = np.zeros(r.shape[0], dtype=SCATTER_DTYPE)
    F.check(lib.b200rt_scatter(scene.device(device), r.ctypes.data, h.ctypes.data, r.shape[0], seed,
                               None if s is None else s.ctypes.data, out.ctypes.data))
    return out


def camera_rays(cam: F.Camera, xy, seed: int = 0, device: int = -1, *, stream=None, with_draws: bool = False):
    """Camera::pixel_ray for jittered pixel coordinates (b200rt_camera_rays): rays float32[n, 6], and with `with_draws`
    also the lens draws each record took (uint32[n]).  `stream`: see _as_stream (None: record i draws from (seed, i, 0))."""
    xy = np.ascontiguousarray(xy, dtype=np.float32)
    s = _as_stream(stream, xy.shape[0])
    out = np.empty((xy.shape[0], 6), dtype=np.float32)
    draws = np.empty(xy.shape[0], dtype=np.uint32) if with_draws else None
    F.check(lib.b200rt_camera_rays(C.byref(cam), xy.ctypes.data, xy.shape[0], seed, None if s is None else s.ctypes.data,
                                   out.ctypes.data, None if draws is None else draws.ctypes.data, device))
    return (out, draws) if with_draws else out


def texture_value(scene: Scene, tex: int, uvp, device: int = -1) -> np.ndarray:
    q = np.ascontiguousarray(uvp, dtype=np.float32)
    out = np.empty((q.shape[0], 3), dtype=np.float32)
    F.check(lib.b200rt_texture_value(scene.device(device), tex, q.ctypes.data, q.shape[0], out.ctypes.data))
    return out


def rng_uniforms(seed: int, a: int, b: int, n: int, device: int = -1) -> np.ndarray:
    out = np.empty(n, dtype=np.float32)
    F.check(lib.b200rt_rng_uniforms(seed, a, b, n, out.ctypes.data, device))
    return out


def fp32_peak(device: int = -1) -> float:
    v = C.c_double()
    F.check(lib.b200rt_fp32_peak(device, C.byref(v)))
    return v.value


def read_peak(nbytes: int, device: int = -1) -> float:
    """Measured read bandwidth in GB/s over a buffer of `nbytes` (48 MiB: the L2 ceiling; 4 GiB: the HBM ceiling)."""
    v = C.c_double()
    F.check(lib.b200rt_read_peak(device, nbytes, C.byref(v)))
    return v.value


def device_count() -> int:
    return lib.b200rt_device_count()
