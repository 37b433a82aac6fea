/*
 * b200rt.h — C ABI of the B200-native path-tracing backend.
 *
 * This is the drop-in boundary for ONE hot path of scottschroeder/shirley-raytracing-rs:
 * the per-pixel path-tracing loop
 *     render_scene (src/main.rs:65-130)
 *       -> render_scanline / ray_color        (src/raytracer/render.rs:17-70)
 *       -> Camera::pixel_ray                  (src/raytracer/camera/mod.rs:98-131)
 *       -> WorkspaceScene::hit_workspace      (src/raytracer/scene/mod.rs:153-163)
 *       -> BboxTree::hit_workspace            (src/raytracer/bvh/bbox_tree.rs:56-91)
 *       -> Material::scatter / Texture::value (src/raytracer/material/...)
 *       -> image::to_image                    (src/raytracer/image.rs:31-44)
 *
 * The reference has no FFI of its own (it is pure Rust); these are the entry points a
 * `gpu` render backend inside src/raytracer would bind (see INTEGRATION.md for the Rust
 * `extern "C"` block).  Everything is plain pointers and sizes.  All input pointers are
 * BORROWED for the duration of the call only; b200rt_scene_create copies what it needs to
 * the device.  Every function returns 0 on success or a negative B200RT_E* code; a
 * thread-local message is available from b200rt_last_error().  Nothing throws or aborts
 * across this boundary, and there is no CPU fallback: without a CUDA device every compute
 * entry point returns B200RT_ECUDA.
 *
 * Arithmetic: the reference computes in f64 (core/math.rs:5); this backend computes in
 * f32 on the device ("dtype": "f32").  Scene data crosses the boundary as f32; the camera
 * crosses as f64 (13 scalars) and is reduced to f32 constants host-side.
 */
#ifndef B200RT_H
#define B200RT_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200RT_ABI_VERSION 1

/* ---- status codes -------------------------------------------------------------------- */
#define B200RT_OK        0
#define B200RT_EINVAL   -1  /* bad argument / malformed scene description                  */
#define B200RT_ECUDA    -2  /* CUDA runtime error (incl. "no device")                      */
#define B200RT_ENOMEM   -3  /* host or device allocation failed                            */
#define B200RT_ESTACK   -4  /* BVH deeper than the fixed device traversal stack            */
#define B200RT_EIO      -5  /* file I/O (PNG writer)                                       */

/* ---- geometry: geometry/object.rs:9-16 (closed enum GeometricObject) ------------------ */
#define B200RT_PRIM_SPHERE   0u  /* geometry/sphere.rs:12-15                                */
#define B200RT_PRIM_RECT_XY  1u  /* Rect<0,1>: d1 = x, d2 = y, plane normal +z  (rect.rs:11) */
#define B200RT_PRIM_RECT_YZ  2u  /* Rect<1,2>: d1 = y, d2 = z, plane normal +x  (rect.rs:12) */
#define B200RT_PRIM_RECT_XZ  3u  /* Rect<0,2>: d1 = x, d2 = z, plane normal +y  (rect.rs:13) */
#define B200RT_PRIM_BOX      4u  /* RectBox  (rect.rs:102-163)                              */

typedef struct B200rtSphere {   /* 16 B, loaded as one float4 */
    float cx, cy, cz, radius;
} B200rtSphere;

typedef struct B200rtRect {     /* 32 B; rect.rs:46-52 */
    float d1_min, d1_max, d2_min, d2_max;
    float offset;               /* plane position on the normal axis */
    uint32_t kind;              /* B200RT_PRIM_RECT_{XY,YZ,XZ} */
    uint32_t _pad[2];
} B200rtRect;

typedef struct B200rtBox {      /* 32 B; RectBox::new(p0, p1), rect.rs:112 */
    float min[3]; float _pad0;
    float max[3]; float _pad1;
} B200rtBox;

/* One entry per scene object, in SceneBuilder::add order (scene/mod.rs:98-109).
 * The index of an entry IS the hit id reported everywhere in this API. */
typedef struct B200rtPrimRef {
    uint32_t type;              /* B200RT_PRIM_* */
    uint32_t index;             /* into spheres[] / rects[] / boxes[] */
} B200rtPrimRef;

/* ---- materials: material/material_type.rs:20-27 (same variant order) ------------------ */
#define B200RT_MAT_METAL          0u  /* metal.rs:10-40      albedo + fuzz (clamped <= 1)   */
#define B200RT_MAT_DIELECTRIC     1u  /* dielectric.rs:10-50 ir                             */
#define B200RT_MAT_LAMBERTIAN     2u  /* lambertian.rs:10-37 texture                        */
#define B200RT_MAT_DIFFUSE_LIGHT  3u  /* lighting.rs:10-29   texture, emits, never scatters */
#define B200RT_MAT_FAIRY_LIGHT    4u  /* lighting.rs:31-67   texture, emits and scatters    */

typedef struct B200rtMaterial { /* 32 B; one per object, indexed by hit id (scene/mod.rs:18-21) */
    uint32_t kind;              /* B200RT_MAT_* */
    int32_t  texture;           /* index into textures[] (Lambertian / lights), else -1 */
    float    albedo[3];         /* Metal only */
    float    param;             /* Metal: fuzz; Dielectric: ir */
    uint32_t _pad[2];
} B200rtMaterial;

/* ---- textures: material/texture/loader.rs:17-28 (TextureLoader, post-dedup) ----------- */
#define B200RT_TEX_SOLID    0u  /* solid.rs:17-21            rgb                            */
#define B200RT_TEX_IMAGE    1u  /* image_texture.rs:34-56    image = index into images[]    */
#define B200RT_TEX_PERLIN   2u  /* perlin/mod.rs:162-184     scalar = scale, image = index into perlin[] */
#define B200RT_TEX_CHECKER  3u  /* checker.rs:27-37          scalar = size, odd/even = child texture indices */

typedef struct B200rtTexture {  /* 32 B */
    uint32_t kind;
    float    rgb[3];
    float    scalar;
    int32_t  odd, even;         /* CHECKER children (must reference LOWER indices: no cycles) */
    int32_t  image;             /* IMAGE: images[] index; PERLIN: perlin[] index */
} B200rtTexture;

typedef struct B200rtImage {    /* decoded RGB8, row 0 = top row of the file, tightly packed */
    uint32_t width, height;
    const uint8_t* rgb8;
} B200rtImage;

/* Perlin tables (perlin/mod.rs:13-18).  The reference draws them from an unseeded RNG and
 * never serialises them (loader.rs:52), so the host supplies them explicitly. */
typedef struct B200rtPerlin {
    float   ranfloat[256][3];   /* un-normalised gradients in [-1,1)^3 */
    uint8_t perm_x[256], perm_y[256], perm_z[256];
} B200rtPerlin;

/* ---- skybox: skybox/mod.rs:11-26 -------------------------------------------------------- */
#define B200RT_SKY_ABOVE 0u
#define B200RT_SKY_FLAT  1u
#define B200RT_SKY_NONE  2u
typedef struct B200rtSkybox { uint32_t kind; float rgb[3]; } B200rtSkybox;

/* ---- flattened scene = SceneBuilder (scene/mod.rs:79-83) after texture dedup ------------ */
typedef struct B200rtSceneDesc {
    uint32_t abi_version;       /* B200RT_ABI_VERSION */
    uint32_t n_prims;     const B200rtPrimRef*  prims;
                          const B200rtMaterial* materials;   /* n_prims entries */
    uint32_t n_spheres;   const B200rtSphere*   spheres;
    uint32_t n_rects;     const B200rtRect*     rects;
    uint32_t n_boxes;     const B200rtBox*      boxes;
    uint32_t n_textures;  const B200rtTexture*  textures;
    uint32_t n_images;    const B200rtImage*    images;
    uint32_t n_perlin;    const B200rtPerlin*   perlin;
    B200rtSkybox skybox;
} B200rtSceneDesc;

/* ---- camera: camera/mod.rs:87-94 (Camera) + :62-69 (CameraPosition) --------------------- */
typedef struct B200rtCamera {
    double   height, width;     /* viewport: 2*tan(vfov/2), aspect*height  (camera/mod.rs:46-50) */
    double   lens_radius;       /* aperture/2; < 0 means None (no lens draw) (camera/mod.rs:51) */
    double   focal_length;
    uint32_t image_width, image_height;   /* Dimmensions (camera/mod.rs:133-137) */
    double   origin[3];
    double   focus_length;      /* pub field; the CLI overwrites it to 10.0 (src/scenes.rs:229) */
    double   w[3], u[3], v[3];
} B200rtCamera;

/* ---- render parameters: RenderSettings (src/argparse.rs:107-123) + sharding ------------- */
#define B200RT_FLAG_COUNT_TRAVERSAL 1u  /* also count BVH node visits / primitive tests (slower) */
#define B200RT_FLAG_ACCUMULATE      2u  /* add to the buffer instead of overwriting (progressive rendering): device API, and
                                           the host API when `accum` is given — its contents are uploaded first and
                                           the RGB8 output is resolved with n = the summed sample count (.w)          */

typedef struct B200rtRenderParams {
    uint32_t samples;           /* per pixel, this call; 0 is coerced to 1 (src/main.rs:75-80) */
    uint32_t sample_offset;     /* index of the first sample (sample-range sharding)           */
    uint32_t max_depth;         /* ray_color's max_depth (render.rs:22), CLI default 50        */
    uint32_t flags;
    uint64_t seed;              /* RNG key; sample s of pixel p depends only on (seed, p, sample_offset+s) */
    uint32_t row_begin, row_end;/* scanlines [begin,end) to render (row 0 = bottom); 0,0 = all */
    uint32_t shard_count;       /* interleaved tile sharding: render tiles t with              */
    uint32_t shard_index;       /*   t % shard_count == shard_index; 0 or 1 = no sharding      */
    int32_t  device;            /* CUDA device ordinal, -1 = current                           */
    uint32_t _pad;
} B200rtRenderParams;

typedef struct B200rtStats {
    uint64_t rays;              /* closest-hit queries = path segments incl. primaries (render.rs:31) */
    uint64_t paths;             /* primary samples                                             */
    uint64_t node_visits;       /* BVH inner-node visits      (only with COUNT_TRAVERSAL)      */
    uint64_t prim_tests;        /* primitive intersection tests (only with COUNT_TRAVERSAL)    */
    uint64_t depth_exhausted;   /* paths that ran out of max_depth (render.rs:30)              */
    double   kernel_ms;         /* device time of the path-tracing kernel(s), CUDA events      */
    double   total_ms;          /* device time incl. copies issued by this call                */
    uint32_t launches;          /* kernels launched by this call                               */
    uint32_t _pad;
    uint64_t diag[8];           /* kernel-version specific lane-utilisation counters (COUNT_TRAVERSAL
                                   only; see DESIGN.md); not part of the parity contract          */
} B200rtStats;

typedef struct B200rtSceneInfo {
    uint32_t n_prims, n_bvh_nodes, bvh_depth, bvh_nodes_in_smem;
    uint64_t device_bytes;
    float    bvh_build_ms;      /* tree construction alone (host wall time, or device time for the device builder) */
    uint32_t bvh_builder;       /* 0 = binned SAH on the host, 1 = linear BVH built on the device (large scenes) */
} B200rtSceneInfo;

typedef struct B200rtScene B200rtScene;    /* opaque, immutable after create */

/* ---- parity-hook records ----------------------------------------------------------------- */
typedef struct B200rtRay { float ox, oy, oz, dx, dy, dz; } B200rtRay;     /* core/vec3.rs:240-244 */

typedef struct B200rtHit {                 /* geometry/hittable.rs:7-14 */
    float   t;
    float   p[3];
    float   n[3];                          /* already face-flipped (hittable.rs:25-28) */
    float   u, v;
    int32_t front_face;
    int32_t id;                            /* hit id, -1 = miss */
} B200rtHit;

typedef struct B200rtScatter {             /* material/mod.rs:14-18 + emitted() */
    B200rtRay ray;                         /* Scatter.direction (a Ray) */
    float   attenuation[3];
    float   emitted[3];                    /* Material::emitted or 0 */
    int32_t scattered;                     /* 1 = Some(scatter), 0 = None */
    uint32_t draws;                        /* RNG draws consumed */
} B200rtScatter;

/* ---- library ------------------------------------------------------------------------------ */
const char* b200rt_last_error(void);
int  b200rt_abi_version(void);
/* Number of visible CUDA devices (0 when there is none / no driver). */
int  b200rt_device_count(void);

/* Replaces SceneBuilder::finalize's BboxTree::new (scene/mod.rs:111-137,
 * bvh/bbox_tree/constructor.rs:9-36): validates the description, builds a BVH (own
 * binned-SAH builder; closest-hit results do not depend on topology), uploads everything
 * to `device` (-1 = current). */
int  b200rt_scene_create(const B200rtSceneDesc* desc, int device, B200rtScene** out);
void b200rt_scene_destroy(B200rtScene* scene);
int  b200rt_scene_info(const B200rtScene* scene, B200rtSceneInfo* out);

/* Replaces the frame loop of render_scene (src/main.rs:85-126): every pixel of the
 * selected rows/tiles gets SUM over `samples` of ray_color(pixel_ray(..)) exactly like
 * render_scanline's `*buf_c = c` (render.rs:59-68).  `accum` is a HOST buffer of
 * image_height*image_width float4 {r,g,b,n}: rgb = sum of radiance, n = number of samples
 * summed; row 0 = bottom of the picture (image.rs:36-38).  Pixels outside the selected
 * rows/tiles are written as zeros.  `stats` may be NULL. */
int  b200rt_render(const B200rtScene* scene, const B200rtCamera* camera,
                   const B200rtRenderParams* params, float* accum, B200rtStats* stats);

/* render_scene's whole product (src/main.rs:85-128 minus the file write): render, then
 * to_image's resolve (image.rs:34-40) on the device, then ONE device->host copy of the
 * W*H*3 RGB8 bytes (top row first).  `accum` may be NULL; if not, the float4 sums are
 * copied back as well. */
int  b200rt_render_rgb8(const B200rtScene* scene, const B200rtCamera* camera,
                        const B200rtRenderParams* params, uint8_t* out_rgb8, float* accum,
                        B200rtStats* stats);

/* Tile-adaptive sampling: every 8x4 tile is rendered until its estimated output error is at most `threshold`.
 * Sampling runs in passes over the tiles still active.  After pass k each of them has
 *     n_k = min(initial_samples * 2^k, max_samples)
 * samples; pass k renders samples [n_{k-1}, n_k) (n_{-1} = 0), offset by params->sample_offset, with the same RNG keying as
 * b200rt_render (sample s of pixel p depends only on (seed, p, sample_offset + s)).  After every pass k >= 1 each active tile's
 * error is estimated from the two independent means of the samples before the pass (n of them, exact sum F) and of the pass
 * (s of them, exact sum P); per pixel and channel c, with every mean clamped at 1 like to_image:
 *     a_c = min(F_c / n, 1)   b_c = min(P_c / s, 1)   m_c = min((F_c + P_c) / (n + s), 1)
 *     sigma_c = |a_c - b_c| * sqrt(n s) / (n + s)                   standard error of the combined mean
 *     e_p = max_c sigma_c / (2 sqrt(max(m_c, 2^-16)))               the same error after to_image's sqrt, 0..1 output units
 *     e_T = max of e_p over the tile's selected pixels
 * A tile stops after pass k when e_T <= threshold or n_k == max_samples; no tile stops before its first estimate, so every
 * selected pixel gets at least min(2 * initial_samples, max_samples) samples.  threshold = 1/255 is about one 8-bit level
 * of standard error.
 *
 * params: seed, max_depth, sample_offset, rows and device as for b200rt_render; `samples` is ignored; COUNT_TRAVERSAL is
 * honoured.  ACCUMULATE, shard_count > 1, initial_samples == 0, max_samples <= initial_samples, a negative or non-finite
 * threshold and a NULL scene, camera, params or adaptive return B200RT_EINVAL.
 * Outputs (each may be NULL; host buffers):
 *   accum       H*W float4 as for b200rt_render, but .w is the pixel's own sample count; pixels outside the rows are zero.
 *               A tile that stopped after n samples equals a plain n-sample b200rt_render of it bit for bit, as long as no
 *               sample's channel exceeds 2e9 / max_samples (the fixed-point clamp is taken for max_samples; every shipped
 *               scene stays far below it).
 *   out_rgb8    the resolve with per-pixel counts: equal to b200rt_resolve_rgb8(accum, W, H, 0, ...).
 *   tile_error  ceil(W/8) * ceil(H/4) floats, tile (tx, ty) covering x in [8tx, 8tx+8), y in [4ty, 4ty+4) (row 0 = bottom,
 *               as in accum): the tile's e_T at its last pass; -1 for tiles with no selected pixel.
 * stats: rays and paths summed over the passes (paths = the sum of .w over the selected pixels), kernel_ms = the summed
 * path-tracing kernel times, total_ms and launches for the whole call.  The call synchronises once per pass to read how many
 * tiles are still active. */
typedef struct B200rtAdaptiveParams {
    uint32_t initial_samples;   /* first pass, every selected tile; >= 1 */
    uint32_t max_samples;       /* no pixel gets more; > initial_samples */
    float    threshold;         /* stop a tile when e_T <= threshold (0..1 output units); >= 0, finite */
    uint32_t _pad;
} B200rtAdaptiveParams;

int  b200rt_render_adaptive(const B200rtScene* scene, const B200rtCamera* camera,
                            const B200rtRenderParams* params, const B200rtAdaptiveParams* adaptive,
                            float* accum, uint8_t* out_rgb8, float* tile_error, B200rtStats* stats);

/* render_scene on SEVERAL GPUs from one host process: `params->samples` is the total per pixel, split into
 * contiguous sample ranges over `devices[0 .. n_devices)` (each gets its own copy of the scene, uploaded by its
 * own host thread); devices[0] sums the per-device buffers inside the resolve through peer access and returns
 * the RGB8 frame.  The devices must be peer-accessible (NVLink / NVSwitch box).  `stats` sums rays / paths and
 * takes the maximum of the kernel times.
 * B200rtMulti is the frame-loop form: the handle owns what does not change between frames — one worker thread,
 * stream, event and accumulation buffer per device, the frame buffer, peer access — so a frame costs only the
 * scene upload, the launches and the copy-back.  b200rt_render_rgb8_multi is the one-shot form: it keeps one
 * handle per device list for the life of the process. */
typedef struct B200rtMulti B200rtMulti;
int  b200rt_multi_create(const int* devices, uint32_t n_devices, B200rtMulti** out);
int  b200rt_multi_render_rgb8(B200rtMulti* multi, const B200rtSceneDesc* desc, const B200rtCamera* camera,
                              const B200rtRenderParams* params, uint8_t* out_rgb8, B200rtStats* stats);
void b200rt_multi_destroy(B200rtMulti* multi);
int  b200rt_render_rgb8_multi(const B200rtSceneDesc* desc, const int* devices, uint32_t n_devices,
                              const B200rtCamera* camera, const B200rtRenderParams* params,
                              uint8_t* out_rgb8, B200rtStats* stats);

/* Same, but `d_accum` is a DEVICE pointer (float4 per pixel) on the scene's device and the
 * work is enqueued on `cuda_stream` (a cudaStream_t, NULL = default stream) without
 * synchronising; stats (if not NULL) are filled by b200rt_render_device_finish. Lets a
 * host keep accumulation buffers resident and combine them across GPUs itself (NCCL). */
int  b200rt_render_device(const B200rtScene* scene, const B200rtCamera* camera,
                          const B200rtRenderParams* params, float* d_accum, void* cuda_stream);
int  b200rt_render_device_finish(const B200rtScene* scene, void* cuda_stream, B200rtStats* stats);

/* Replaces to_image's pixel loop (image.rs:34-40) + Color::to_pixel (core/color.rs:31-38):
 * out[(H-1-j)*W + i] = sat_u8(sqrt(accum[j][i].rgb / n) * 255.999), n = accum[j][i].w when
 * samples == 0 else `samples`.  Host buffers. `out` is W*H*3 bytes, top row first. */
int  b200rt_resolve_rgb8(const float* accum, uint32_t width, uint32_t height, uint32_t samples,
                         uint8_t* out_rgb8, int device);
int  b200rt_resolve_rgb8_device(const float* d_accum, uint32_t width, uint32_t height,
                                uint32_t samples, uint8_t* d_out_rgb8, void* cuda_stream);

/* Multi-GPU, one process per GPU (SURVEY.md §8e): the cross-GPU sum of sample-range-sharded
 * accumulation buffers FUSED into to_image's resolve (image.rs:34-40).  Every process creates
 * its accumulation buffer with b200rt_peer_buffer_create (cudaMalloc + an IPC handle, 64 opaque
 * bytes the host exchanges however it likes, e.g. torch.distributed.all_gather_object), opens
 * the other ranks' handles, renders into its own buffer (b200rt_render_device), synchronises
 * the ranks' streams (a barrier), and then resolves a band of rows [row_begin, row_end) from
 * ALL buffers at once: out[(H-1-j)*W + i] = sat_u8(sqrt(sum_r accum_r[j][i].rgb / n) * 255.999),
 * summed in the order given (deterministic bytes).  d_out_rgb8 is the W*H*3 frame — normally a
 * peer pointer to the root rank's frame buffer, so the bands of all ranks assemble there over
 * NVLink without an intermediate reduced float buffer.  n = `samples` (total over ranks), or
 * the summed .w when samples == 0.  (0, 0) selects all rows. */
#define B200RT_PEER_HANDLE_BYTES 64
int  b200rt_peer_buffer_create(int device, size_t bytes, void** d_ptr, uint8_t handle[B200RT_PEER_HANDLE_BYTES]);
int  b200rt_peer_buffer_open(int device, const uint8_t handle[B200RT_PEER_HANDLE_BYTES], void** d_ptr);
int  b200rt_peer_buffer_close(int device, void* d_ptr);      /* a pointer from _open  */
int  b200rt_peer_buffer_destroy(int device, void* d_ptr);    /* a pointer from _create */
/* Stream-ordered cross-GPU barrier over peer memory, no library collective: each rank creates a flag array of
 * B200RT_PEER_FLAG_BYTES with b200rt_peer_buffer_create (zeroed) and opens its peers'.  _signal writes `epoch`
 * into slot [slot][my_rank] of EVERY rank's array (system-scope release after the stream's earlier work);
 * _wait blocks the stream until all ranks' epochs in [slot] of the OWN array reached `epoch` (acquire).
 * slot 0: "my accumulation buffer is complete" (before the fused resolve), slot 1: "I have finished reading"
 * (before the next frame overwrites the buffers, and before rank 0 reads the assembled frame).  A peer that
 * never arrives ends the wait after timeout_ms (0 = 10 s) and is reported by b200rt_peer_timed_out
 * (*out = 1 + rank, 0 = none) instead of hanging the device; the host must treat that frame as failed. */
#define B200RT_PEER_FLAG_BYTES 256
int  b200rt_peer_signal_device(uint32_t* const* d_flag_arrays, uint32_t n_peers, uint32_t my_rank,
                               uint32_t slot, uint32_t epoch, void* cuda_stream);
int  b200rt_peer_wait_device(uint32_t* d_my_flags, uint32_t n_peers, uint32_t slot, uint32_t epoch,
                             uint32_t timeout_ms, void* cuda_stream);
int  b200rt_peer_timed_out(uint32_t* d_my_flags, uint32_t* out);   /* synchronises; reading a time-out also clears it */
/* d_my_flags: this rank's flag array (or NULL).  When given, a resolve enqueued after a flag wait that timed out
 * stores NOTHING (an incomplete peer buffer never becomes a frame); b200rt_peer_timed_out then reports the rank. */
int  b200rt_resolve_peers_rgb8_device(const float* const* d_accums, uint32_t n_peers,
                                      uint32_t width, uint32_t height, uint32_t samples,
                                      uint32_t row_begin, uint32_t row_end,
                                      uint8_t* d_out_rgb8, const uint32_t* d_my_flags, void* cuda_stream);

/* Replaces RgbImage::save_with_format(.., Png) (image.rs:42): 8-bit RGB PNG via zlib. */
int  b200rt_write_png(const char* path, const uint8_t* rgb8, uint32_t width, uint32_t height);
/* Same encoder into a malloc'ed buffer; release with b200rt_free. */
int  b200rt_encode_png(const uint8_t* rgb8, uint32_t width, uint32_t height, uint8_t** out_bytes, size_t* out_len);
void b200rt_free(void* p);

/* ---- parity hooks (each runs a CUDA kernel; used by tests/ against oracle/) ------------- */

/* K1: Scene/BboxTree::hit_workspace over a ray array (bvh/bbox_tree.rs:56-91).
 * ids[i] = hit id or -1; hits may be NULL. Interval is inclusive on both ends like
 * sphere.rs:41-46; among exactly equal t the highest id wins.  stats (may be NULL): rays and kernel_ms always;
 * node_visits / prim_tests only when `hits` is requested too (ids-only calls run without the counters). */
int  b200rt_closest_hit(const B200rtScene* scene, const B200rtRay* rays, size_t n,
                        float t_min, float t_max, int32_t* ids, B200rtHit* hits,
                        B200rtStats* stats);

/* Aabb::hit2 (bvh/aabb.rs:62-79) in f32: boxes[i] = {min xyz, max xyz}; out[i] = 0/1. */
int  b200rt_aabb_hit(const float* boxes6, const B200rtRay* rays, size_t n,
                     float t_min, float t_max, uint8_t* out, int device);

/* K4: Material::scatter + ::emitted (material_type.rs:50-79) for hit records `hits`
 * produced by incoming rays `rays`; the material is materials[hits[i].id]. Record i draws
 * its random numbers from the stream b200rt_rng(seed, i, 0) (see below). */
int  b200rt_scatter(const B200rtScene* scene, const B200rtRay* rays, const B200rtHit* hits,
                    size_t n, uint64_t seed, B200rtScatter* out);

/* Camera::pixel_ray (camera/mod.rs:98-131) for pixel coordinates xy[2*i], xy[2*i+1]
 * (already jittered); record i draws the lens sample from stream b200rt_rng(seed, i, 0). */
int  b200rt_camera_rays(const B200rtCamera* camera, const float* xy, size_t n, uint64_t seed,
                        B200rtRay* out, int device);

/* Texture::value (material/texture/mod.rs:8-10) of textures[tex] at (u, v, p). */
int  b200rt_texture_value(const B200rtScene* scene, int32_t tex, const float* uvp5, size_t n,
                          float* out_rgb);

/* The first `n` uniform [0,1) draws of stream (seed, a, b) — documents the RNG so the
 * oracle can replay it:  key = hash(seed, a, b) -> (state, inc);  per draw
 *   state = state * 747796405 + inc;  w = ((state >> ((state >> 28) + 4)) ^ state) * 277803737;
 *   w ^= w >> 22;  uniform = (w >> 8) * 2^-24.
 * In b200rt_render: a = pixel index (row * width + column), b = sample index. */
int  b200rt_rng_uniforms(uint64_t seed, uint32_t a, uint32_t b, size_t n, float* out, int device);

/* Measured FP32 issue ceiling of the device: FFMA-chain microbenchmark; returns
 * lane-instructions per second (FMA counted once) in *out. Roofline denominator. */
int  b200rt_fp32_peak(int device, double* lane_instr_per_s);
/* Measured read bandwidth (GB/s) over a device buffer of `bytes` (>= 1 MiB), float4 loads through L2 (.cg): a buffer well
 * inside the L2 (e.g. 48 MiB) gives the L2 ceiling, a multi-GB one the HBM ceiling.  Roofline denominators for scenes whose
 * BVH lives in global memory. */
int  b200rt_read_peak(int device, size_t bytes, double* gb_per_s);

#ifdef __cplusplus
}
#endif
#endif /* B200RT_H */
