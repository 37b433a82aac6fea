"""ctypes binding of include/b200rt.h and include/b200rt_host.h.

The library is the product: if ``libb200rt.so`` is missing this module raises at import
time — there is no Python/NumPy fallback for any compute entry point.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200RT_LIB") or os.path.join(_HERE, "libb200rt.so")   # B200RT_LIB: an alternative build (A/B runs of kernel variants)

# ---- status codes --------------------------------------------------------------------------
OK, EINVAL, ECUDA, ENOMEM, ESTACK, EIO = 0, -1, -2, -3, -4, -5
ABI_VERSION = 1

PRIM_SPHERE, PRIM_RECT_XY, PRIM_RECT_YZ, PRIM_RECT_XZ, PRIM_BOX = range(5)
MAT_METAL, MAT_DIELECTRIC, MAT_LAMBERTIAN, MAT_DIFFUSE_LIGHT, MAT_FAIRY_LIGHT = range(5)
TEX_SOLID, TEX_IMAGE, TEX_PERLIN, TEX_CHECKER = range(4)
SKY_ABOVE, SKY_FLAT, SKY_NONE = range(3)
FLAG_COUNT_TRAVERSAL, FLAG_ACCUMULATE = 1, 2


class Sphere(C.Structure):
    _fields_ = [("cx", C.c_float), ("cy", C.c_float), ("cz", C.c_float), ("radius", C.c_float)]


class Rect(C.Structure):
    _fields_ = [("d1_min", C.c_float), ("d1_max", C.c_float), ("d2_min", C.c_float), ("d2_max", C.c_float),
                ("offset", C.c_float), ("kind", C.c_uint32), ("_pad", C.c_uint32 * 2)]


class Box(C.Structure):
    _fields_ = [("min", C.c_float * 3), ("_pad0", C.c_float), ("max", C.c_float * 3), ("_pad1", C.c_float)]


class PrimRef(C.Structure):
    _fields_ = [("type", C.c_uint32), ("index", C.c_uint32)]


class Material(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("texture", C.c_int32), ("albedo", C.c_float * 3), ("param", C.c_float),
                ("_pad", C.c_uint32 * 2)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("rgb", C.c_float * 3), ("scalar", C.c_float), ("odd", C.c_int32),
                ("even", C.c_int32), ("image", C.c_int32)]


class Image(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("rgb8", C.POINTER(C.c_uint8))]


class Perlin(C.Structure):
    _fields_ = [("ranfloat", (C.c_float * 3) * 256), ("perm_x", C.c_uint8 * 256), ("perm_y", C.c_uint8 * 256),
                ("perm_z", C.c_uint8 * 256)]


class Skybox(C.Structure):
    _fields_ = [("kind", C.c_uint32), ("rgb", C.c_float * 3)]


class SceneDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32),
                ("n_prims", C.c_uint32), ("prims", C.POINTER(PrimRef)), ("materials", C.POINTER(Material)),
                ("n_spheres", C.c_uint32), ("spheres", C.POINTER(Sphere)),
                ("n_rects", C.c_uint32), ("rects", C.POINTER(Rect)),
                ("n_boxes", C.c_uint32), ("boxes", C.POINTER(Box)),
                ("n_textures", C.c_uint32), ("textures", C.POINTER(Texture)),
                ("n_images", C.c_uint32), ("images", C.POINTER(Image)),
                ("n_perlin", C.c_uint32), ("perlin", C.POINTER(Perlin)),
                ("skybox", Skybox)]


class Camera(C.Structure):
    _fields_ = [("height", C.c_double), ("width", C.c_double), ("lens_radius", C.c_double), ("focal_length", C.c_double),
                ("image_width", C.c_uint32), ("image_height", C.c_uint32), ("origin", C.c_double * 3),
                ("focus_length", C.c_double), ("w", C.c_double * 3), ("u", C.c_double * 3), ("v", C.c_double * 3)]


class RenderParams(C.Structure):
    _fields_ = [("samples", C.c_uint32), ("sample_offset", C.c_uint32), ("max_depth", C.c_uint32), ("flags", C.c_uint32),
                ("seed", C.c_uint64), ("row_begin", C.c_uint32), ("row_end", C.c_uint32), ("shard_count", C.c_uint32),
                ("shard_index", C.c_uint32), ("device", C.c_int32), ("_pad", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [("rays", C.c_uint64), ("paths", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64),
                ("depth_exhausted", C.c_uint64), ("kernel_ms", C.c_double), ("total_ms", C.c_double),
                ("launches", C.c_uint32), ("_pad", C.c_uint32), ("diag", C.c_uint64 * 8)]


class AdaptiveParams(C.Structure):
    _fields_ = [("initial_samples", C.c_uint32), ("max_samples", C.c_uint32), ("threshold", C.c_float), ("_pad", C.c_uint32)]


class SceneInfo(C.Structure):
    _fields_ = [("n_prims", C.c_uint32), ("n_bvh_nodes", C.c_uint32), ("bvh_depth", C.c_uint32),
                ("bvh_nodes_in_smem", C.c_uint32), ("device_bytes", C.c_uint64), ("bvh_build_ms", C.c_float), ("bvh_builder", C.c_uint32)]


class Ray(C.Structure):
    _fields_ = [("ox", C.c_float), ("oy", C.c_float), ("oz", C.c_float), ("dx", C.c_float), ("dy", C.c_float), ("dz", C.c_float)]


class Hit(C.Structure):
    _fields_ = [("t", C.c_float), ("p", C.c_float * 3), ("n", C.c_float * 3), ("u", C.c_float), ("v", C.c_float),
                ("front_face", C.c_int32), ("id", C.c_int32)]


class Scatter(C.Structure):
    _fields_ = [("ray", Ray), ("attenuation", C.c_float * 3), ("emitted", C.c_float * 3), ("scattered", C.c_int32),
                ("draws", C.c_uint32)]


# Every symbol declared in include/b200rt.h and include/b200rt_host.h: (restype, argtypes)
_P = C.POINTER
SIGNATURES = {
    # b200rt.h
    "b200rt_last_error": (C.c_char_p, []),
    "b200rt_abi_version": (C.c_int, []),
    "b200rt_device_count": (C.c_int, []),
    "b200rt_scene_create": (C.c_int, [_P(SceneDesc), C.c_int, _P(C.c_void_p)]),
    "b200rt_scene_destroy": (None, [C.c_void_p]),
    "b200rt_scene_info": (C.c_int, [C.c_void_p, _P(SceneInfo)]),
    "b200rt_render": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, _P(Stats)]),
    "b200rt_render_rgb8": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p, _P(Stats)]),
    "b200rt_render_adaptive": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), _P(AdaptiveParams), C.c_void_p, C.c_void_p,
                                         C.c_void_p, _P(Stats)]),
    "b200rt_render_rgb8_multi": (C.c_int, [_P(SceneDesc), _P(C.c_int), C.c_uint32, _P(Camera), _P(RenderParams), C.c_void_p, _P(Stats)]),
    "b200rt_render_device": (C.c_int, [C.c_void_p, _P(Camera), _P(RenderParams), C.c_void_p, C.c_void_p]),
    "b200rt_render_device_finish": (C.c_int, [C.c_void_p, C.c_void_p, _P(Stats)]),
    "b200rt_resolve_rgb8": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]),
    "b200rt_resolve_rgb8_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "b200rt_peer_buffer_create": (C.c_int, [C.c_int, C.c_size_t, _P(C.c_void_p), C.c_void_p]),
    "b200rt_peer_buffer_open": (C.c_int, [C.c_int, C.c_void_p, _P(C.c_void_p)]),
    "b200rt_peer_buffer_close": (C.c_int, [C.c_int, C.c_void_p]),
    "b200rt_peer_buffer_destroy": (C.c_int, [C.c_int, C.c_void_p]),
    "b200rt_peer_signal_device": (C.c_int, [_P(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "b200rt_peer_wait_device": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "b200rt_peer_timed_out": (C.c_int, [C.c_void_p, _P(C.c_uint32)]),
    "b200rt_resolve_peers_rgb8_device": (C.c_int, [_P(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200rt_multi_create": (C.c_int, [_P(C.c_int), C.c_uint32, _P(C.c_void_p)]),
    "b200rt_multi_render_rgb8": (C.c_int, [C.c_void_p, _P(SceneDesc), _P(Camera), _P(RenderParams), C.c_void_p, _P(Stats)]),
    "b200rt_multi_destroy": (None, [C.c_void_p]),
    "b200rt_write_png": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32]),
    "b200rt_encode_png": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _P(C.c_void_p), _P(C.c_size_t)]),
    "b200rt_free": (None, [C.c_void_p]),
    "b200rt_closest_hit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float, C.c_void_p, C.c_void_p, _P(Stats)]),
    "b200rt_aabb_hit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_float, C.c_float, C.c_void_p, C.c_int]),
    "b200rt_scatter": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p]),
    "b200rt_camera_rays": (C.c_int, [_P(Camera), C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p, C.c_int]),
    "b200rt_texture_value": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200rt_rng_uniforms": (C.c_int, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_size_t, C.c_void_p, C.c_int]),
    "b200rt_fp32_peak": (C.c_int, [C.c_int, _P(C.c_double)]),
    "b200rt_read_peak": (C.c_int, [C.c_int, C.c_size_t, _P(C.c_double)]),
    # b200rt_host.h
    "b200rt_host_last_error": (C.c_char_p, []),
    "b200rt_host_scene_from_json": (C.c_int, [C.c_char_p, C.c_size_t, C.c_uint64, _P(C.c_void_p)]),
    "b200rt_host_scene_to_json": (C.c_int, [C.c_void_p, _P(C.c_void_p), _P(C.c_size_t)]),
    "b200rt_host_scene_named": (C.c_int, [C.c_char_p, C.c_uint64, C.c_uint32, _P(C.c_void_p)]),
    "b200rt_host_scene_destroy": (None, [C.c_void_p]),
    "b200rt_host_scene_desc": (_P(SceneDesc), [C.c_void_p]),
    "b200rt_host_register_image": (C.c_int, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "b200rt_host_decode_image": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_uint32), _P(C.c_uint32), _P(C.c_void_p)]),
    "b200rt_host_decode_jpeg": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_uint32), _P(C.c_uint32), _P(C.c_void_p)]),
    "b200rt_host_checkpoint_save": (C.c_int, [C.c_char_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64]),
    "b200rt_host_checkpoint_load": (C.c_int, [C.c_char_p, _P(C.c_uint32), _P(C.c_uint32), _P(C.c_uint32), _P(C.c_uint64), _P(C.c_void_p)]),
    "b200rt_host_camera": (C.c_int, [_P(C.c_double), _P(C.c_double), _P(C.c_double), C.c_double, C.c_double, C.c_double,
                                     C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, _P(Camera)]),
    "b200rt_host_default_camera": (C.c_int, [C.c_uint32, C.c_double, C.c_double, C.c_double, C.c_uint32, C.c_uint32, _P(Camera)]),
    "b200rt_host_render_scene": (C.c_int, [C.c_void_p, _P(Camera), C.c_uint32, C.c_uint32, C.c_uint64, C.c_int, C.c_char_p,
                                           C.c_void_p, _P(Stats)]),
}


def load(path: str = LIB_PATH) -> C.CDLL:
    if not os.path.exists(path):
        raise ImportError(
            f"{path} not found: build it with `make lib` (or __graft_entry__.build()). "
            "shirley_raytracing_rs_b200 has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here = header/library mismatch
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()


class B200rtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200rt error {code}: {msg}")
        self.code = code


def check(rc: int, host: bool = False) -> None:
    if rc != OK:
        msg = (lib.b200rt_host_last_error() if host else lib.b200rt_last_error()) or b""
        raise B200rtError(rc, msg.decode("utf-8", "replace"))
