"""ctypes mirror of include/functracer_b200.h (the C ABI the F# shim binds with P/Invoke).

Every Structure here must stay field-for-field identical to the header; tests/test_abi.py
checks sizes and that the shared library exports every declared symbol.
"""
import ctypes as C

ABI_VERSION = 4

# ftb_status
OK = 0
ERR_BAD_ARG = -1
ERR_BAD_SCENE = -2
ERR_UNSUPPORTED = -3
ERR_HIT_OVERFLOW = -4
ERR_CUDA = -5
ERR_OOM = -6
ERR_NO_DEVICE = -7

# ftb_node_kind (Scene.fs:33-53)
NODE_PRIMITIVE, NODE_TRANSFORM, NODE_MATERIAL, NODE_TEXTURE, NODE_HUESHIFT, NODE_IGNORELIGHT, \
    NODE_GROUP, NODE_UNION, NODE_INTERSECT, NODE_SUBTRACT, NODE_EXCLUDE = range(11)
# ftb_prim_kind (Scene.fs:8-18)
PRIM_BSPMESH, PRIM_CIRCLE, PRIM_SQUARE, PRIM_CUBE, PRIM_SPHERE, PRIM_PLANE, PRIM_CONE, \
    PRIM_SOLIDCYLINDER, PRIM_CYLINDER, PRIM_TRIANGLE = range(10)
PRIM_NAMES = ["bspMesh", "circle", "square", "cube", "sphere", "plane", "cone", "solidCylinder",
              "cylinder", "triangle"]
TEX_IMAGE, TEX_GRID, TEX_SCALE, TEX_ROTATE = range(4)
LIGHT_DIRECTIONAL, LIGHT_SOFT_DIRECTIONAL, LIGHT_POINT = range(3)
SAMPLING_JITTER, SAMPLING_CORNER = 0, 1
PRECISION_FP32, PRECISION_FP64_VERIFY = 0, 1
OUT_RGB_F64, OUT_RGB_F32, OUT_RGBA8 = 0, 1, 2
TILE_W = TILE_H = 16
TILE_PIXELS = TILE_W * TILE_H


class Node(C.Structure):
    _fields_ = [("kind", C.c_int32), ("a", C.c_int32), ("b", C.c_int32), ("reserved", C.c_int32)]


class Transform(C.Structure):
    _fields_ = [("m2w", C.c_double * 12), ("w2m", C.c_double * 12)]


class Material(C.Structure):
    _fields_ = [("colour", C.c_double * 3), ("roughness", C.c_double), ("reflectance", C.c_double),
                ("shineyness", C.c_double), ("apply_lighting", C.c_int32), ("reserved", C.c_int32)]


class Texture(C.Structure):
    _fields_ = [("kind", C.c_int32), ("inner", C.c_int32), ("image", C.c_int32), ("reserved", C.c_int32),
                ("p", C.c_double * 6)]


class Image(C.Structure):
    _fields_ = [("rgb24", C.POINTER(C.c_uint8)), ("width", C.c_int32), ("height", C.c_int32)]


class BspNode(C.Structure):
    _fields_ = [("aabb_min", C.c_double * 3), ("aabb_max", C.c_double * 3), ("left", C.c_int32),
                ("right", C.c_int32)]


class BspLeaf(C.Structure):
    _fields_ = [("tri_first", C.c_int32), ("tri_count", C.c_int32)]


class Mesh(C.Structure):
    _fields_ = [("root", C.c_int32), ("reserved", C.c_int32)]


class Light(C.Structure):
    _fields_ = [("kind", C.c_int32), ("samples", C.c_int32), ("v", C.c_double * 3),
                ("falloff", C.c_double * 3), ("scatter_rad", C.c_double), ("colour", C.c_double * 3)]


class SceneDesc(C.Structure):
    _fields_ = [
        ("root", C.c_int32), ("n_nodes", C.c_int32), ("nodes", C.POINTER(Node)),
        ("n_children", C.c_int32), ("children", C.POINTER(C.c_int32)),
        ("n_transforms", C.c_int32), ("transforms", C.POINTER(Transform)),
        ("n_materials", C.c_int32), ("materials", C.POINTER(Material)),
        ("n_textures", C.c_int32), ("textures", C.POINTER(Texture)),
        ("n_images", C.c_int32), ("images", C.POINTER(Image)),
        ("n_meshes", C.c_int32), ("meshes", C.POINTER(Mesh)),
        ("n_bsp_nodes", C.c_int32), ("bsp_nodes", C.POINTER(BspNode)),
        ("n_bsp_leaves", C.c_int32), ("bsp_leaves", C.POINTER(BspLeaf)),
        ("n_triangles", C.c_int32), ("triangles", C.POINTER(C.c_double)),
        ("n_lights", C.c_int32), ("lights", C.POINTER(Light)),
    ]


class Camera(C.Structure):
    _fields_ = [("o", C.c_double * 3), ("look_at", C.c_double * 3), ("up", C.c_double * 3),
                ("fov_y_rad", C.c_double), ("aspect_ratio", C.c_double), ("has_focus", C.c_int32),
                ("reserved", C.c_int32), ("focal_length", C.c_double), ("aperture_rad", C.c_double)]


class RenderParams(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("sampling", C.c_int32),
                ("jitter_xy", C.POINTER(C.c_double)), ("recursion_limit", C.c_int32),
                ("precision", C.c_int32), ("seed", C.c_uint64), ("out_format", C.c_int32),
                ("shard_index", C.c_int32), ("shard_count", C.c_int32), ("n_gpus", C.c_int32),
                ("collect_stats", C.c_int32), ("band_index", C.c_int32), ("band_count", C.c_int32),
                ("reserved", C.c_int32)]


class DebugOut(C.Structure):
    _fields_ = [("prim_id", C.POINTER(C.c_int32)), ("sub_id", C.POINTER(C.c_int32)),
                ("t", C.POINTER(C.c_double))]


class HitOut(C.Structure):
    """ftb_hit_out: the planes of a nearest-hit query (any pointer may be NULL = not wanted)."""
    _fields_ = [("t", C.POINTER(C.c_double)), ("prim_id", C.POINTER(C.c_int32)), ("sub_id", C.POINTER(C.c_int32)),
                ("p", C.POINTER(C.c_double)), ("normal", C.POINTER(C.c_double)), ("colour", C.POINTER(C.c_double)),
                ("surface", C.POINTER(C.c_double))]


class PathOut(C.Structure):
    """ftb_path_out: the planes of a path query (any pointer may be NULL = not wanted)."""
    _fields_ = [("levels", C.POINTER(C.c_int32)), ("colour", C.POINTER(C.c_double)), ("ray_od", C.POINTER(C.c_double)),
                ("weight", C.POINTER(C.c_double)), ("hit", HitOut), ("intensity", C.POINTER(C.c_double)),
                ("light_dir", C.POINTER(C.c_double)), ("light_colour", C.POINTER(C.c_double))]


class Stats(C.Structure):
    _fields_ = [("primary_rays", C.c_uint64), ("shadow_rays", C.c_uint64), ("reflection_rays", C.c_uint64),
                ("shaded_hits", C.c_uint64), ("leaf_tests", C.c_uint64 * 10),
                ("transformed_leaf_tests", C.c_uint64), ("bsp_nodes_visited", C.c_uint64),
                ("bound_tests", C.c_uint64), ("csg_ops", C.c_uint64), ("flops", C.c_double),
                ("kernel_ms", C.c_double), ("total_ms", C.c_double), ("kernel_launches", C.c_int32),
                ("hit_overflow", C.c_int32)]

    def as_dict(self):
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if hasattr(v, "__len__") else v
        return d


# Every symbol include/functracer_b200.h declares.
EXPORTS = [
    "ftb_abi_version", "ftb_device_count", "ftb_last_error", "ftb_scene_create", "ftb_scene_destroy",
    "ftb_render", "ftb_tile_buffer_bytes", "ftb_render_tiles_device", "ftb_assemble_device",
    "ftb_shade_rays", "ftb_band_rows", "ftb_assemble_rows_device", "ftb_host_copy_begin", "ftb_host_copy_finish",
    "ftb_check_overflow", "ftb_scene_build_info", "ftb_render_window", "ftb_render_window_tiles_device",
    "ftb_intersect_rays", "ftb_occluded_rays", "ftb_intersect_rays_device", "ftb_occluded_rays_device",
    "ftb_intersect_all_rays", "ftb_intersect_all_rays_device", "ftb_trace_paths", "ftb_trace_paths_device",
    "ftb_frame_rays", "ftb_frame_rays_device", "ftb_shade_samples", "ftb_shade_samples_device",
]
