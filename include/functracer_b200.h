/* functracer_b200.h — C ABI of the B200 render-loop replacement for FuncTracer.
 *
 * The reference (antonburger/FuncTracer, F#) has no FFI today; this header is the seam the
 * F# shim binds with P/Invoke (see INTEGRATION.md).  It replaces, for the render loop only:
 *
 *   Shading.shade            FuncTracer/Shading.fs:141-147   -> ftb_shade_rays / ftb_render
 *   SamplingStrategy.generateRays / blendPixels   FuncTracer/Image.fs:100-116,128-144
 *                                                            -> ftb_render (fused on device)
 *   Scene.intersect (SceneGraph -> closure)   FuncTracer/Scene.fs:67-104
 *                                                            -> ftb_scene_create (SceneGraph -> device SoA)
 *   call site                FuncTracer/Program.fs:54-64
 *
 * Everything is plain C: blittable structs, cdecl, no callbacks, no exceptions, no ownership
 * transfer (every create copies what it needs; the caller frees its own arrays).
 * All reals are IEEE double at the boundary (the reference's `float`).  Return value 0 = OK,
 * negative = ftb_status error; ftb_last_error() gives a thread-local message.
 *
 * The scene is handed over as the reference's own data form: the SceneGraph discriminated
 * union (Scene.fs:33-53) serialised into a flat node array, plus side tables for the
 * payloads.  Lowering (matrix pre-composition per leaf, static surface resolution, CSG
 * program linearisation, SoA upload) happens inside the library.
 */
#ifndef FUNCTRACER_B200_H
#define FUNCTRACER_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FTB_ABI_VERSION 4

typedef enum ftb_status {
    FTB_OK = 0,
    FTB_ERR_BAD_ARG = -1,      /* null pointer, bad size, bad enum */
    FTB_ERR_BAD_SCENE = -2,    /* index out of range, cycle, malformed graph */
    FTB_ERR_UNSUPPORTED = -3,  /* legal grammar the device path does not implement (documented) */
    FTB_ERR_HIT_OVERFLOW = -4, /* a CSG operand produced more crossings than the per-ray hit stack holds */
    FTB_ERR_CUDA = -5,
    FTB_ERR_OOM = -6,
    FTB_ERR_NO_DEVICE = -7
} ftb_status;

/* ---- SceneGraph (Scene.fs:33-53) ------------------------------------------------------ */

typedef enum ftb_node_kind {
    FTB_NODE_PRIMITIVE = 0,   /* a = ftb_prim_kind, b = payload (mesh index | triangle index | 0) */
    FTB_NODE_TRANSFORM = 1,   /* a = index into transforms[], b = child node   (SceneFunction(Transform t, g)) */
    FTB_NODE_MATERIAL = 2,    /* a = index into materials[],  b = child node */
    FTB_NODE_TEXTURE = 3,     /* a = index into textures[],   b = child node */
    FTB_NODE_HUESHIFT = 4,    /* a unused,                    b = child node (angle is ignored, CommonTypes.fs:90) */
    FTB_NODE_IGNORELIGHT = 5, /* a unused,                    b = child node */
    FTB_NODE_GROUP = 6,       /* a = first index into children[], b = child count (may be 0) */
    FTB_NODE_UNION = 7,       /* a = node of operand A, b = node of operand B */
    FTB_NODE_INTERSECT = 8,
    FTB_NODE_SUBTRACT = 9,
    FTB_NODE_EXCLUDE = 10
} ftb_node_kind;

/* Scene.fs:8-18, same order */
typedef enum ftb_prim_kind {
    FTB_PRIM_BSPMESH = 0,
    FTB_PRIM_CIRCLE = 1,
    FTB_PRIM_SQUARE = 2,
    FTB_PRIM_CUBE = 3,
    FTB_PRIM_SPHERE = 4,
    FTB_PRIM_PLANE = 5,
    FTB_PRIM_CONE = 6,
    FTB_PRIM_SOLIDCYLINDER = 7,
    FTB_PRIM_CYLINDER = 8,
    FTB_PRIM_TRIANGLE = 9
} ftb_prim_kind;

typedef struct ftb_node {
    int32_t kind;
    int32_t a;
    int32_t b;
    int32_t reserved;
} ftb_node;

/* One SceneFunction(Transform t, _) node.  Both matrices are built on the HOST by the
 * reference's own Transform.matrix (Transform.fs:55-71) so that host and device consume
 * identical numbers; row-major 3x4 (the 4th row of every reference matrix is 0 0 0 1).
 *   m2w = matrix t            (modelToWorld, Transform.fs:81)
 *   w2m = matrix (inverse t)  (worldToModel, Transform.fs:82); normalToWorld = transpose(w2m) (:83) */
typedef struct ftb_transform {
    double m2w[12];
    double w2m[12];
} ftb_transform;

/* Ray.fs:4-10 */
typedef struct ftb_material {
    double colour[3];
    double roughness;
    double reflectance;
    double shineyness;
    int32_t apply_lighting; /* the parser always builds materials from mattWhite => 1 (SceneParser.fs:99-105) */
    int32_t reserved;
} ftb_material;

/* Scene.fs:47-53 (Texture / TextureFunction) */
typedef enum ftb_texture_kind {
    FTB_TEX_IMAGE = 0,  /* image = index into images[] */
    FTB_TEX_GRID = 1,   /* p[0..2] = colour1, p[3..5] = colour2 (Texture.fs:24-29) */
    FTB_TEX_SCALE = 2,  /* TextureFunction(inner, Scale(p[0], p[1]))  (Texture.fs:14-16) */
    FTB_TEX_ROTATE = 3  /* TextureFunction(inner, Rotate angle): p[0] = angle rad, p[1] = cos, p[2] = sin
                           as produced by the host's matrix (rotate unitY angle) (Texture.fs:18-22) */
} ftb_texture_kind;

typedef struct ftb_texture {
    int32_t kind;
    int32_t inner; /* SCALE / ROTATE: index of the wrapped texture */
    int32_t image; /* IMAGE: index into images[] */
    int32_t reserved;
    double p[6];
} ftb_texture;

/* Decoded Rgb24 pixel data exactly as Textures/Image.fs:24-26 holds it (row 0 = top). */
typedef struct ftb_image {
    const uint8_t* rgb24;
    int32_t width;
    int32_t height;
} ftb_image;

/* BspMesh.fs:12-19 surfaced as data.  Child links: >= 0 -> index into bsp_nodes[] (Branch),
 * < 0 -> ~link indexes bsp_leaves[] (Leaf). */
typedef struct ftb_bsp_node {
    double aabb_min[3];
    double aabb_max[3];
    int32_t left;
    int32_t right;
} ftb_bsp_node;

typedef struct ftb_bsp_leaf {
    int32_t tri_first; /* into triangles[], in the leaf's own sequence order */
    int32_t tri_count;
} ftb_bsp_leaf;

typedef struct ftb_mesh {
    int32_t root; /* same link encoding; a depth-0 mesh is one bare leaf (BspMesh.fs:95-97) */
    int32_t reserved;
} ftb_mesh;

/* Light.fs:7-14.  Directions arrive normalised (Light.fs:19-23). */
typedef enum ftb_light_kind {
    FTB_LIGHT_DIRECTIONAL = 0,
    FTB_LIGHT_SOFT_DIRECTIONAL = 1,
    FTB_LIGHT_POINT = 2
} ftb_light_kind;

typedef struct ftb_light {
    int32_t kind;
    int32_t samples;    /* soft directional */
    double v[3];        /* direction (directional kinds) or position (point) */
    double falloff[3];  /* constant, linear, quadratic (point) */
    double scatter_rad; /* soft directional */
    double colour[3];
} ftb_light;

typedef struct ftb_scene_desc {
    int32_t root; /* node index of Scene.objects (the top-level Group, SceneParser.fs:354) */
    int32_t n_nodes;
    const ftb_node* nodes;
    int32_t n_children;
    const int32_t* children; /* Group child node indices, in list order */
    int32_t n_transforms;
    const ftb_transform* transforms;
    int32_t n_materials;
    const ftb_material* materials;
    int32_t n_textures;
    const ftb_texture* textures;
    int32_t n_images;
    const ftb_image* images;
    int32_t n_meshes;
    const ftb_mesh* meshes;
    int32_t n_bsp_nodes;
    const ftb_bsp_node* bsp_nodes;
    int32_t n_bsp_leaves;
    const ftb_bsp_leaf* bsp_leaves;
    int32_t n_triangles;
    const double* triangles; /* 9 doubles each: a, b, c (Triangle.fs:6) */
    int32_t n_lights;
    const ftb_light* lights; /* Scene.lights, in file order */
} ftb_scene_desc;

/* ---- camera / sampling (Image.fs:9-17, 67-150) ---------------------------------------- */

typedef struct ftb_camera {
    double o[3];
    double look_at[3];
    double up[3]; /* already normalised by the parser (SceneParser.fs:280) */
    double fov_y_rad;
    double aspect_ratio;
    int32_t has_focus;
    int32_t reserved;
    double focal_length;
    double aperture_rad;
} ftb_camera;

typedef enum ftb_sampling { FTB_SAMPLING_JITTER = 0, FTB_SAMPLING_CORNER = 1 } ftb_sampling;
typedef enum ftb_precision { FTB_PRECISION_FP32 = 0, FTB_PRECISION_FP64_VERIFY = 1 } ftb_precision;
typedef enum ftb_out_format {
    FTB_OUT_RGB_F64 = 0, /* 3 doubles per pixel, blended, un-clamped: Bitmap.pixels (Image.fs:30) */
    FTB_OUT_RGB_F32 = 1, /* 3 floats per pixel, same values narrowed */
    FTB_OUT_RGBA8 = 2    /* Image.write's quantisation applied on device (Image.fs:36-40): clamp, *255, truncate; A = 255 */
} ftb_out_format;

typedef struct ftb_render_params {
    int32_t width;  /* resH */
    int32_t height; /* resV */
    int32_t spp;    /* samples per pixel (jitter mode) */
    int32_t sampling;
    const double* jitter_xy; /* 2*spp offsets in the unit disc, drawn on the HOST exactly as
                                Image.fs:101-105 does; required in jitter mode */
    int32_t recursion_limit; /* Shading.fs:142 uses 8 */
    int32_t precision;
    uint64_t seed;      /* counter-based RNG seed for soft shadows / depth of field (DESIGN.md) */
    int32_t out_format;
    int32_t shard_index; /* tile sharding across GPUs/ranks: this call renders tiles t with */
    int32_t shard_count; /*   t % shard_count == shard_index; 0 or 1 = whole frame            */
    int32_t n_gpus;      /* ftb_render only: in-process multi-GPU, 0/1 = current device only  */
    int32_t collect_stats; /* 1 = run the counting variant of the kernel (slower) */
    int32_t band_index;  /* ftb_render_tiles_device only: render just the tiles of band band_index of band_count    */
    int32_t band_count;  /*   horizontal bands of tile rows (ftb_band_rows gives a band's pixel rows); 0/1 = all    */
    int32_t reserved;
} ftb_render_params;

/* Optional per-primary-sample debug planes (W*H*spp each, sample-major within pixel,
 * pixels row-major; a window's planes hold its own samples only, see ftb_render_window), the device analogue of Program.printIntersectionAt (Program.fs:33-49).
 * prim_id = depth-first index of the PRIMITIVE node instance that produced the nearest hit
 * (-1 = miss); sub_id = face 0..5 for cubes (bottom, top, left, right, front, back;
 * Cube.fs:24), part 0..2 for solidCylinder (top, bottom, sides; Cylinder.fs:29), index into
 * triangles[] for meshes, else 0. */
typedef struct ftb_debug_out {
    int32_t* prim_id;
    int32_t* sub_id;
    double* t;
} ftb_debug_out;

typedef struct ftb_stats {
    uint64_t primary_rays;
    uint64_t shadow_rays;
    uint64_t reflection_rays; /* unique reflection rays (SURVEY.md 8d) */
    uint64_t shaded_hits;
    uint64_t leaf_tests[10];  /* by ftb_prim_kind; a cube and a solidCylinder count once each, mesh triangles tested
                                 count under FTB_PRIM_TRIANGLE */
    uint64_t transformed_leaf_tests;
    uint64_t bsp_nodes_visited; /* nodes of the device's mesh index (a BVH over the BSP's triangles) visited */
    uint64_t bound_tests;     /* object-level bound tests (no counterpart in the reference) */
    uint64_t csg_ops;
    double flops;             /* algorithmic flops by the SURVEY.md 8(d) table (+ 17 per bound test, 5 when answered from the common-origin table) */
    double kernel_ms;         /* device time of the render kernel(s) */
    double total_ms;          /* wall time of the call */
    int32_t kernel_launches;
    int32_t hit_overflow;
} ftb_stats;

typedef struct ftb_scene ftb_scene; /* opaque */

int ftb_abi_version(void);
int ftb_device_count(void);
const char* ftb_last_error(void);

/* Copies every array in desc; uploads the lowered SoA scene to the current CUDA device
 * (and lazily to the other devices ftb_render is asked to use). */
int ftb_scene_create(const ftb_scene_desc* desc, ftb_scene** out);
void ftb_scene_destroy(ftb_scene* scene);

/* How the mesh index of the scene was built (BspMesh.fs:30-65 is the reference's own, lazily clipped tree; the
 * device traverses its own index over the same triangles, built on the GPU at create time): whether the device
 * build was used, the device time of its kernels and the wall time including transfers (0 without meshes). */
int ftb_scene_build_info(const ftb_scene* scene, int32_t* bvh_on_device, double* bvh_build_ms, double* bvh_total_ms);

/* Host-buffer entry point = the drop-in for Program.fs:54-64.  out is caller-allocated:
 * W*H pixels in params->out_format, row-major (y, then x), blended (Image.fs:112-116 /
 * 134-144) and un-clamped unless RGBA8.  dbg and stats may be NULL.
 *
 * out may be ordinary pageable memory (a GC-pinned .NET array, a std::vector, a numpy array) or CUDA
 * page-locked memory: the frame is rendered in up to four bands of tile rows, ALL of them queued before
 * the first byte is copied, and every finished band is downloaded while the later bands render, so only
 * the last band's copy is exposed.  FTB_OUT_RGBA8 is what Image.write keeps of a frame (Image.fs:35-44:
 * clamp, * 255, truncate) at 1/6 of the bytes of FTB_OUT_RGB_F64.
 *
 * One scene holds ONE frame in flight per device: the per-device scratch (tile queue counter, jitter table,
 * tile order) is shared by all calls on that scene; concurrent frames need separate ftb_scene objects. */
int ftb_render(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params,
               void* out, const ftb_debug_out* dbg, ftb_stats* stats);

/* Device-buffer entry points (for callers that own device memory and a stream, e.g. one
 * process per GPU under torch.distributed).  All pointers are device pointers on the
 * current device; stream is a cudaStream_t (0 = default stream).
 *
 * ftb_render_tiles_device renders this shard's tiles into a tile-major FP32/FP64 buffer
 * (ftb_tile_buffer_bytes gives its size: n_local_tiles * FTB_TILE_PIXELS * 3 reals);
 * ftb_assemble_device turns shard_count such buffers (device pointers, all on the current
 * device, e.g. after an NCCL gather) into the final row-major frame in out_format. */
#define FTB_TILE_W 16
#define FTB_TILE_H 16
#define FTB_TILE_PIXELS (FTB_TILE_W * FTB_TILE_H)

int64_t ftb_tile_buffer_bytes(const ftb_render_params* params);
int ftb_render_tiles_device(ftb_scene* scene, const ftb_camera* camera,
                            const ftb_render_params* params, void* d_tiles,
                            const ftb_debug_out* d_dbg, ftb_stats* stats, void* stream);
int ftb_assemble_device(const ftb_render_params* params, const void* const* d_tile_buffers,
                        void* d_out, void* stream);

/* Banded variants for callers that overlap the frame's download with its rendering (what ftb_render does
 * inside one process): ftb_band_rows gives the pixel rows [*y0, *y1) of band band_index of band_count
 * (whole tile rows; later bands are smaller so that the last, exposed copy is short);
 * ftb_render_tiles_device with params->band_count > 1 renders only that band's tiles of the shard;
 * ftb_assemble_rows_device assembles only rows [y0, y1) of the frame (d_out still addresses row 0). */
int ftb_band_rows(const ftb_render_params* params, int band_index, int band_count, int* y0, int* y1);
int ftb_assemble_rows_device(const ftb_render_params* params, const void* const* d_tile_buffers,
                             void* d_out, int y0, int y1, void* stream);

/* Windows: the pixel rectangle [x0, x1) x [y0, y1) of the frame that params->width x params->height
 * describes (0 <= x0 < x1 <= width, 0 <= y0 < y1 <= height; anything else is FTB_ERR_BAD_ARG), e.g. a crop,
 * a one-pixel probe, or a rectangle of the caller's own tiling of a frame.  A window renders exactly what the
 * whole frame renders there, bit for bit, in every out_format and precision, debug planes included: its
 * rays, RNG keys and blend order are the whole frame's.  Only the outputs are packed to the window:
 *   - out holds (x1-x0)*(y1-y0) pixels, row-major within the window;
 *   - the debug planes hold (x1-x0)*(y1-y0)*spp entries, sample-major within a pixel, pixels row-major within
 *     the window; in corner sampling the window's sample grid is the corners [x0, x1] x [y0, y1], so they
 *     hold (x1-x0+1)*(y1-y0+1) entries.
 * ftb_render_window takes everything ftb_render takes (n_gpus, pageable or page-locked out, stats).
 * ftb_render_window_tiles_device takes everything ftb_render_tiles_device takes (shard_index / shard_count,
 * band_index / band_count) over the window's tiles.  A window's tile buffer IS the tile buffer of a frame of
 * the window's size: ftb_tile_buffer_bytes, ftb_band_rows, ftb_assemble_device and ftb_assemble_rows_device
 * called with a copy of params whose width / height are x1-x0 / y1-y0 size it, band it and assemble it.
 * ftb_render and ftb_render_tiles_device are the window (0, 0, width, height) of these two. */
int ftb_render_window(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params,
                      int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                      void* out, const ftb_debug_out* dbg, ftb_stats* stats);
int ftb_render_window_tiles_device(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params,
                                   int32_t x0, int32_t y0, int32_t x1, int32_t y1,
                                   void* d_tiles, const ftb_debug_out* d_dbg, ftb_stats* stats, void* stream);

/* Device -> host copy of a finished band behind the work already queued on `stream` (current device).
 * A page-locked destination makes the call asynchronous; with a pageable one it returns when that band has
 * arrived (the driver stages it at link speed) - so queue ALL rendering and assembly first, then begin the
 * copies in the order the bands finish: the GPU renders band c + 1 while the host sits in the copy of band c.
 * ftb_host_copy_finish waits for every copy begun on the scene for the current device; after it returns the
 * data is in place. */
int ftb_host_copy_begin(ftb_scene* scene, const void* d_src, void* host_dst, int64_t bytes, void* stream);
int ftb_host_copy_finish(ftb_scene* scene);

/* The device entry points never synchronise, so a CSG hit-stack or mesh-stack overflow inside
 * ftb_render_tiles_device cannot be returned by that call: this one waits for `stream`, returns
 * FTB_ERR_HIT_OVERFLOW if any frame rendered on the current device since the last check overflowed
 * (FTB_OK otherwise) and clears the flag.  ftb_render and ftb_shade_rays check by themselves. */
int ftb_check_overflow(ftb_scene* scene, void* stream);

/* Literal Shading.shade replacement (Shading.fs:141): caller supplies n explicit rays
 * (o.xyz, d.xyz per ray, i.e. what generateRays + depthOfFieldJitter produced in F#) and
 * receives n colours in the same order; blending stays with the caller.  Host buffers.
 * dbg planes, if given, hold n entries. */
int ftb_shade_rays(ftb_scene* scene, const double* rays_od, int64_t n,
                   const ftb_render_params* params, double* out_rgb,
                   const ftb_debug_out* dbg, ftb_stats* stats);

/* ---- ray queries: Scene.closest (Scene.fs:112-118) and Scene.lightIsBocked (Scene.fs:119-121) ----------------------
 * n caller-supplied rays (o.xyz, d.xyz doubles per ray, as for ftb_shade_rays), answered by the renderer's own trace.
 *   - Rays are traced exactly as given: no 1e-4 slightOffset (that belongs to Shading, not to Scene.closest), and d need
 *     not be unit length; t is in units of d.
 *   - Nearest: the smallest t >= 0, the first in enumeration order on ties, as the renderer decides it.  The record is the
 *     fragment the renderer shades (in FP32 a hit on a planar leaf is projected back onto its plane); prim_id / sub_id are
 *     those of the debug planes of ftb_debug_out.  A miss: t = -1, prim_id = -1, sub_id = 0, every other requested plane 0.
 *   - Occlusion: blocked[i] = 1 iff some surface with applyLighting crosses ray i at 0 <= t < max_t[i] (max_t may be +inf),
 *     else 0.  No leaf is skipped: callers offset shadow-ray origins as the reference does (by 1e-4 n).
 *   - params: only precision and collect_stats are read.  The counting kernel counts nearest queries as primary_rays and
 *     occlusion queries as shadow_rays.  Calls run on the current device; a multi-GPU caller splits the batch itself.
 *   - A query uses the scene's per-device control block, as a frame does: one frame or query in flight per scene and device.
 *   - NULL scene or params, n < 0, or NULL rays / max_t / blocked with n > 0: FTB_ERR_BAD_ARG; n = 0 is OK; no CUDA device:
 *     FTB_ERR_NO_DEVICE.  A CSG hit-stack overflow: FTB_ERR_HIT_OVERFLOW from the host entry points (which then leave the
 *     caller's arrays unwritten), from
 *     ftb_check_overflow after the device entry points (which never synchronise, except to fill stats). */
typedef struct ftb_hit_out { /* any pointer may be NULL = not wanted; n entries of the given width each */
    double* t;        /* n    nearest t >= 0 in units of d; -1 on a miss                               */
    int32_t* prim_id; /* n    as in ftb_debug_out: -1 on a miss                                        */
    int32_t* sub_id;  /* n    as ftb_debug_out                                                         */
    double* p;        /* 3n   world hit point, as the shader receives it                               */
    double* normal;   /* 3n   world normal after normalToWorld and the CSG flip                        */
    double* colour;   /* 3n   surface colour after textures and hue shifts                             */
    double* surface;  /* 4n   roughness, reflectance, shineyness, apply_lighting (0 / 1)               */
} ftb_hit_out;

/* Host buffers; synchronous.  out may be NULL (nothing wanted but stats). */
int ftb_intersect_rays(ftb_scene* scene, const double* rays_od, int64_t n, const ftb_render_params* params,
                       const ftb_hit_out* out, ftb_stats* stats);
int ftb_occluded_rays(ftb_scene* scene, const double* rays_od, const double* max_t, int64_t n,
                      const ftb_render_params* params, int32_t* blocked, ftb_stats* stats);
/* The same on device pointers of the current device, queued on stream (a cudaStream_t, 0 = default stream). */
int ftb_intersect_rays_device(ftb_scene* scene, const double* d_rays_od, int64_t n, const ftb_render_params* params,
                              const ftb_hit_out* d_out, ftb_stats* stats, void* stream);
int ftb_occluded_rays_device(ftb_scene* scene, const double* d_rays_od, const double* d_max_t, int64_t n,
                             const ftb_render_params* params, int32_t* d_blocked, ftb_stats* stats, void* stream);

/* ---- crossing queries: Scene.intersect (Scene.fs:67-104), every crossing of a ray with the scene, sorted by t -----------
 * n caller-supplied rays as above (o.xyz d.xyz, traced exactly as given, no slightOffset; t in units of d, so the segment
 * from a to b is the ray (a, b - a) with t_max = 1).
 *   - Ray i's crossings are the entries of Scene.intersect's list with t_min <= t < t_max.  t_min = -INFINITY gives the whole
 *     list, including the crossings behind the origin (they set Csg.constructedSolid's inside state) and the t = 0 crossing
 *     Plane.fs gives a ray parallel to a plane from its front side; t_min = 0 gives what lies ahead.
 *   - counts[i] = the number of such crossings; it may exceed max_hits.
 *   - Order: sorted by t, equal t in Scene.intersect's order (Seq.sortBy (fun h -> h.t), the order Scene.closest picks
 *     from): the first crossing with t >= 0 is the one ftb_intersect_rays returns.
 *   - The first min(counts[i], max_hits) crossings are written.  The planes of ftb_hit_out are max_hits entries wide per ray:
 *     entry (i, k) is at i * max_hits + k (times the plane's width: 3 for p, normal, colour, 4 for surface).  Each entry is
 *     the record ftb_intersect_rays gives, built for that crossing: t, prim_id, sub_id, p, normal (after the CSG flip),
 *     colour, surface.  Unused slots read as a miss: t = -1, prim_id = -1, sub_id = 0, 0 in every other plane.
 *   - out may be NULL (counts only); any plane pointer may be NULL = not wanted (left untouched).
 *   - params: only precision and collect_stats are read; the counting kernel counts every ray as a primary ray.
 *   - Bad arguments, checked before any device is looked for: FTB_ERR_BAD_ARG for a NULL scene or params, n < 0, NULL rays
 *     or counts with n > 0, max_hits outside 1 .. FTB_MAX_CROSSINGS, t_min or t_max NaN, or t_min >= t_max.  n = 0 is OK;
 *     no CUDA device: FTB_ERR_NO_DEVICE.
 *   - A CSG hit-stack overflow is reported as by the other queries (the host entry then leaves the caller's arrays
 *     unwritten); one frame or query in flight per scene and device; the device entry synchronises only to fill stats. */
#define FTB_MAX_CROSSINGS 64
int ftb_intersect_all_rays(ftb_scene* scene, const double* rays_od, int64_t n, int32_t max_hits, double t_min, double t_max,
                           const ftb_render_params* params, const ftb_hit_out* out, int32_t* counts, ftb_stats* stats);
int ftb_intersect_all_rays_device(ftb_scene* scene, const double* d_rays_od, int64_t n, int32_t max_hits, double t_min,
                                  double t_max, const ftb_render_params* params, const ftb_hit_out* d_out, int32_t* d_counts,
                                  ftb_stats* stats, void* stream);

/* ---- path queries: why a ray has its colour (Shading.getColourForRay, Shading.fs:109-147) ----------------------------------
 * n caller-supplied rays as for ftb_shade_rays (o.xyz d.xyz).  Each is shaded as ftb_shade_rays shades it, and every level
 * (bounce) of getColourForRay is reported: its ray, nearest hit and weight, and per light the shadow intensity, the light
 * direction and the colour shadeLight gives.  D = params->recursion_limit + 1 level entries per ray, L = the scene's light count:
 * entry (i, k) is at i * D + k, entry (i, k, l) at (i * D + k) * L + l, each times the plane's width.
 *   - Rays and keys: the level-0 ray and every reflected ray get the 1e-4 slightOffset, and hit.t is measured along the offset
 *     ray (as the debug planes of ftb_debug_out measure it).  Soft lights draw from ftb_rng.h with params->seed, depth
 *     recursion_limit - limit and sample key sample_keys[i]; NULL sample_keys means key i, which is what ftb_shade_rays uses.
 *     So a frame sample's primary ray with key (py * gw + px) * spp + s gives that sample's path.
 *   - Colour: colour[i] is the sum the renderer forms: per level, local = 0, then local += light_colour[l] in light order, then
 *     colour += W * local; reflecting multiplies W by L * reflectance.  In FP64 this sum, colour and ftb_shade_rays' output
 *     for the same ray and key are bit-identical.  In FP32 the query runs the generic kernel where ftb_shade_rays may run the
 *     scene's specialised one, so the two agree to FP32 rounding, not bit for bit.
 *   - Levels: levels[i] counts the nearest-hit rays traced (1 .. D).  A level that misses reads t = -1, prim_id = -1,
 *     sub_id = 0 and 0 in every other hit plane and every light plane; its ray and weight are written.  Entries after
 *     levels[i] read as a miss with weight 0 and a zero ray.  With L = 0 nothing is shaded or reflected: level 0 is recorded
 *     and the colour is 0.
 *   - Shadow rays that are not traced: an unlit surface, or an Oren-Nayar surface without a specular term, reports intensity 1
 *     (its colour does not depend on it); a soft light with 0 samples reports NaN, as the reference computes 0 / 0.
 *   - params: only precision, seed, recursion_limit and collect_stats are read.  The counting kernel counts primary, shadow
 *     and reflection rays and shaded hits as ftb_shade_rays' counting kernel does for the same rays; leaf and bound tests also
 *     agree unless a frame's common-origin bound table answers some of ftb_shade_rays' bound tests (scenes of 8 or more
 *     top-level items with point lights), which this query does not use.
 *   - Bad arguments, checked before any device is looked for: FTB_ERR_BAD_ARG for a NULL scene or params, n < 0, NULL rays
 *     with n > 0, a bad precision, or recursion_limit outside 0 .. FTB_MAX_PATH_LEVELS - 1.  n = 0 is OK; no CUDA device:
 *     FTB_ERR_NO_DEVICE.
 *   - A hit-stack overflow is reported as by the other queries (the host entry then leaves the caller's arrays unwritten);
 *     one frame or query in flight per scene and device; the device entry synchronises only to fill stats. */
#define FTB_MAX_PATH_LEVELS 64
typedef struct ftb_path_out {  /* any pointer may be NULL = not wanted (left untouched) */
    int32_t* levels;           /* n      levels traced, 1 .. D                                                        */
    double* colour;            /* 3n     the ray's colour: ftb_shade_rays' value for this ray and key                 */
    double* ray_od;            /* 6nD    each level's ray (o.xyz d.xyz) before slightOffset                           */
    double* weight;            /* nD     the level's running weight W                                                 */
    ftb_hit_out hit;           /* nD each the level's nearest hit, planes as in ftb_hit_out                           */
    double* intensity;         /* nDL    shadow intensity of light l at level k                                       */
    double* light_dir;         /* 3nDL   lightDirection (Shading.fs:44-48) at the hit point                           */
    double* light_colour;      /* 3nDL   shadeLight's colour for light l (specular + diffuse, or the unlit surface
                                         colour); the reflection is in the next level's W                             */
} ftb_path_out;
int ftb_trace_paths(ftb_scene* scene, const double* rays_od, const uint64_t* sample_keys, int64_t n,
                    const ftb_render_params* params, const ftb_path_out* out, ftb_stats* stats);
int ftb_trace_paths_device(ftb_scene* scene, const double* d_rays_od, const uint64_t* d_sample_keys, int64_t n,
                           const ftb_render_params* params, const ftb_path_out* d_out, ftb_stats* stats, void* stream);

/* ---- a frame's own samples: SamplingStrategy.generateRays / blendPixels (Image.fs:100-116) with the rays in the caller's hands ----
 * ftb_frame_rays writes the primary ray and RNG key of every sample of the window [x0, x1) x [y0, y1) of the frame camera + params
 * describe, exactly as the render kernel generates them:
 *   - entries in the debug planes' order and count (see ftb_render_window): jitter sampling (x1-x0)*(y1-y0)*spp entries, sample-major
 *     within a pixel, pixels row-major within the window; corner sampling the (x1-x0+1)*(y1-y0+1) corner grid;
 *   - rays_od: o.xyz d.xyz before slightOffset and after depth-of-field jitter, the kernel's own values widened to double (FP32 rays
 *     narrow back exactly); sample_keys: (py * gw + px) * spp + s, gw the frame's sample-grid width (width, or width + 1 for corners);
 *   - params: only width, height, spp, sampling, jitter_xy, precision and seed are read, and checked as ftb_render_window checks them
 *     (the window too), before any device is looked for; either output pointer may be NULL.
 * ftb_shade_samples shades n_pixels * spp caller-supplied rays (sample s of pixel i is ray i * spp + s) and blends each pixel as
 * ftb_render blends a jitter-mode pixel: Array.average in sample order, in the same passes and fold segments a frame of that spp uses
 * in the same kernel variant.  Each ray is shaded as ftb_shade_rays shades it, with the RNG key sample_keys[i * spp + s]
 * (NULL: the ray's index i * spp + s; with spp = 1 that is what ftb_shade_rays uses).
 *   - out: n_pixels pixels in params->out_format (RGBA8: Image.write's quantisation); dbg, if given, holds n_pixels * spp entries per
 *     plane, as ftb_shade_rays' debug planes do; planes not asked for are not touched.
 *   - params: only spp (>= 1), precision, seed, recursion_limit, out_format and collect_stats are read.  sampling is not: corner
 *     frames blend across pixels.  The variant is picked from the scene's features, as for ftb_shade_rays.
 *   - Contract: shading a window's ftb_frame_rays output with its keys and the same params gives ftb_render_window's result for that
 *     window bit for bit, in every out_format and in the debug planes.  Always in FP64; in FP32 whenever the frame runs the variant this
 *     call runs.  A depth-of-field frame adds FT_RNG to the scene's features and may run another variant: its FP32 pixels then agree
 *     only to FP32 rounding.
 *   - The counting kernel counts primary, shadow and reflection rays and shaded hits as the frame's counting kernel does for the same
 *     samples (the frame adds its clear tiles' samples and the shadow rays it skips on lit ground tiles, as it counts them).
 *   - Bad arguments, checked before any device is looked for: FTB_ERR_BAD_ARG for a NULL scene or params, n_pixels < 0, spp < 1,
 *     NULL rays or out with n_pixels > 0, more than 0x7fffff00 pixels or n_pixels * spp past ftb_shade_rays' ray limit, a bad precision
 *     or out_format.  n_pixels = 0 is OK; no CUDA device: FTB_ERR_NO_DEVICE.
 *   - A hit-stack overflow is reported as by the queries (the host entry then leaves the caller's arrays unwritten); one frame or query
 *     in flight per scene and device; the device entries synchronise only to fill stats. */
int ftb_frame_rays(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params,
                   int32_t x0, int32_t y0, int32_t x1, int32_t y1, double* rays_od, uint64_t* sample_keys);
int ftb_frame_rays_device(ftb_scene* scene, const ftb_camera* camera, const ftb_render_params* params,
                          int32_t x0, int32_t y0, int32_t x1, int32_t y1, double* d_rays_od, uint64_t* d_sample_keys,
                          void* stream);
int ftb_shade_samples(ftb_scene* scene, const double* rays_od, const uint64_t* sample_keys, int64_t n_pixels,
                      const ftb_render_params* params, void* out, const ftb_debug_out* dbg, ftb_stats* stats);
int ftb_shade_samples_device(ftb_scene* scene, const double* d_rays_od, const uint64_t* d_sample_keys, int64_t n_pixels,
                             const ftb_render_params* params, void* d_out, const ftb_debug_out* d_dbg, ftb_stats* stats,
                             void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FUNCTRACER_B200_H */
