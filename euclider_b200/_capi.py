"""ctypes mirror of include/euclider_b200.h (the C ABI of libeuclider_b200.so).

The library is the product; this file only declares its structs and prototypes.  There is no
Python/CPU rendering fallback: if the shared library (or a CUDA device) is missing, the calls
fail loudly.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

EUCL_MAX_DIM = 4
EUCL_MAX_LEVELS = 64
EUCL_IPC_HANDLE_BYTES = 64

c_double4 = C.c_double * EUCL_MAX_DIM
c_int4 = C.c_int32 * EUCL_MAX_DIM


class EuclPrim(C.Structure):
    _fields_ = [("kind", C.c_int32), ("_pad", C.c_int32), ("v0", c_double4), ("v1", c_double4),
                ("s0", C.c_double), ("s1", C.c_double)]


class EuclNode(C.Structure):
    _fields_ = [("op", C.c_int32), ("prim", C.c_int32), ("first", C.c_int32), ("_pad", C.c_int32)]


class EuclEntity(C.Structure):
    _fields_ = [("node_first", C.c_int32), ("node_root", C.c_int32), ("material", C.c_int32), ("surface", C.c_int32)]


class EuclMaterial(C.Structure):
    _fields_ = [("kind", C.c_int32), ("transform_first", C.c_int32), ("n_transforms", C.c_int32), ("_pad", C.c_int32)]


class EuclTransform(C.Structure):
    _fields_ = [("fwd_first", c_int4), ("fwd_len", c_int4), ("inv_first", c_int4), ("inv_len", c_int4)]


class EuclExprOp(C.Structure):
    _fields_ = [("op", C.c_int32), ("arg", C.c_int32), ("value", C.c_double)]


class EuclSurface(C.Structure):
    _fields_ = [("ratio_op", C.c_int32), ("refl_op", C.c_int32), ("thr_op", C.c_int32), ("color_first", C.c_int32),
                ("color_len", C.c_int32), ("_pad", C.c_int32), ("ratio_a", C.c_double), ("ratio_b", C.c_double),
                ("thr_a", C.c_double)]


class EuclColorOp(C.Structure):
    _fields_ = [("op", C.c_int32), ("i0", C.c_int32), ("f", C.c_double * 12)]


class EuclMappedTexture(C.Structure):
    _fields_ = [("uv_kind", C.c_int32), ("filter", C.c_int32), ("texture", C.c_int32), ("_pad", C.c_int32),
                ("center", c_double4)]


class EuclTexture(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("texel_offset", C.c_uint64)]


class EuclCamera(C.Structure):
    _fields_ = [("dim", C.c_int32), ("max_depth", C.c_uint32), ("fov_deg", C.c_uint32), ("_pad", C.c_uint32),
                ("location", c_double4), ("forward", c_double4), ("up", c_double4), ("left", c_double4)]

    def copy(self) -> "EuclCamera":
        out = EuclCamera()
        C.memmove(C.byref(out), C.byref(self), C.sizeof(EuclCamera))
        return out


class EuclFrame(C.Structure):
    _fields_ = [("camera", EuclCamera), ("time_seconds", C.c_double)]


class EuclAovs(C.Structure):
    _fields_ = [("depth", C.c_void_p), ("position", C.c_void_p), ("normal", C.c_void_p), ("segments", C.c_void_p),
                ("levels", C.c_void_p)]


class EuclRays(C.Structure):
    _fields_ = [("origins", C.c_void_p), ("directions", C.c_void_p), ("n", C.c_uint32), ("width", C.c_uint32),
                ("max_depth", C.c_uint32), ("pipeline", C.c_int32), ("time_seconds", C.c_double), ("profile", C.c_int32),
                ("_pad", C.c_int32)]


class EuclTreeNode(C.Structure):
    _fields_ = [("parent", C.c_int32), ("level", C.c_int32), ("kind", C.c_int32), ("medium", C.c_int32),
                ("hit_entity", C.c_int32), ("exiting", C.c_int32), ("flags", C.c_uint32), ("surface_rgba8", C.c_uint32),
                ("ratio", C.c_double), ("t", C.c_double), ("origin", c_double4), ("direction", c_double4),
                ("normal", c_double4), ("color", C.c_double * 4)]


class EuclTreeQuery(C.Structure):
    _fields_ = [("items", C.c_void_p), ("n_items", C.c_uint32), ("capacity", C.c_uint32), ("nodes", C.c_void_p),
                ("counts", C.c_void_p)]


class EuclFlatScene(C.Structure):
    _fields_ = [("dim", C.c_int32),
                ("n_prims", C.c_int32), ("n_nodes", C.c_int32), ("n_entities", C.c_int32),
                ("n_materials", C.c_int32), ("n_transforms", C.c_int32), ("n_expr_ops", C.c_int32),
                ("n_surfaces", C.c_int32), ("n_color_ops", C.c_int32), ("n_mapped_textures", C.c_int32),
                ("n_textures", C.c_int32), ("background", C.c_int32),
                ("prims", C.POINTER(EuclPrim)), ("nodes", C.POINTER(EuclNode)),
                ("entities", C.POINTER(EuclEntity)), ("materials", C.POINTER(EuclMaterial)),
                ("transforms", C.POINTER(EuclTransform)), ("expr_ops", C.POINTER(EuclExprOp)),
                ("surfaces", C.POINTER(EuclSurface)), ("color_ops", C.POINTER(EuclColorOp)),
                ("mapped_textures", C.POINTER(EuclMappedTexture)), ("textures", C.POINTER(EuclTexture)),
                ("texels", C.POINTER(C.c_uint8)), ("texel_bytes", C.c_uint64),
                ("perlin_perm", C.c_uint8 * 256), ("camera", EuclCamera)]


class EuclRenderOpts(C.Structure):
    _fields_ = [("width", C.c_uint32), ("height", C.c_uint32), ("time_seconds", C.c_double),
                ("band_rows", C.c_uint32), ("band_rank", C.c_uint32), ("band_world", C.c_uint32),
                ("pipeline", C.c_int32), ("compact_rows", C.c_int32), ("want_hit_ids", C.c_int32),
                ("profile", C.c_int32), ("_pad", C.c_int32)]


class EuclStats(C.Structure):
    _fields_ = [("pixels", C.c_uint64), ("segments", C.c_uint64), ("nodes", C.c_uint64),
                ("level_counts", C.c_uint64 * EUCL_MAX_LEVELS), ("levels", C.c_uint32), ("retries", C.c_uint32),
                ("launches", C.c_uint32), ("ray_grouping", C.c_uint32), ("ms_total", C.c_float), ("ms_raygen", C.c_float),
                ("ms_intersect", C.c_float), ("ms_shade", C.c_float), ("ms_resolve", C.c_float), ("graph_replays", C.c_uint32)]


# enums (values from the header)
EUCL_OK = 0
EUCL_PIPELINE_WAVEFRONT = 0
EUCL_PIPELINE_MEGAKERNEL = 1
EUCL_PRECISION_F64, EUCL_PRECISION_F32 = 0, 1
EUCL_TREE_ROOT, EUCL_TREE_TRANSMITTED, EUCL_TREE_REFLECTED = range(3)
EUCL_TREE_BACKGROUND, EUCL_TREE_SURFACE, EUCL_TREE_OPAQUE, EUCL_TREE_NO_DESTINATION, EUCL_TREE_UNDEFINED, EUCL_TREE_CHECKERBOARD = (
    1, 2, 4, 8, 16, 32)
EUCL_TREE_MAX_ITEMS = 65536
EUCL_TREE_MAX_NODES = 1 << 24
PRIM_VOID, PRIM_SPHERE, PRIM_HYPERPLANE, PRIM_HALFSPACE, PRIM_CYLINDER = range(5)
CSG_LEAF, CSG_UNION, CSG_INTERSECTION, CSG_COMPLEMENT, CSG_SYMDIFF = range(5)
MAT_VACUUM, MAT_LINEAR_SPACE = range(2)
(BLEND_RATIO, BLEND_OVER, BLEND_INSIDE, BLEND_OUTSIDE, BLEND_ATOP, BLEND_XOR, BLEND_PLUS, BLEND_MULTIPLY,
 BLEND_SCREEN, BLEND_OVERLAY, BLEND_DARKEN, BLEND_LIGHTEN, BLEND_DODGE, BLEND_BURN, BLEND_HARD_LIGHT,
 BLEND_SOFT_LIGHT, BLEND_DIFFERENCE, BLEND_EXCLUSION) = range(18)

STATUS_NAMES = {
    0: "EUCL_OK", -1: "EUCL_ERR_INVALID_ARGUMENT", -10: "EUCL_ERR_PARSE_NO_DESERIALIZER",
    -11: "EUCL_ERR_PARSE_SYNTAX", -12: "EUCL_ERR_PARSE_MISSING_TYPE", -13: "EUCL_ERR_PARSE_INVALID_CONSTRUCTOR",
    -14: "EUCL_ERR_PARSE_MISSING_FIELD", -15: "EUCL_ERR_PARSE_TYPE_MISMATCH", -16: "EUCL_ERR_PARSE_CUSTOM",
    -20: "EUCL_ERR_TEXTURE_MISSING", -21: "EUCL_ERR_SCENE_LIMIT", -30: "EUCL_ERR_CUDA",
    -31: "EUCL_ERR_OUT_OF_MEMORY", -32: "EUCL_ERR_NO_DEVICE",
}

# every symbol include/euclider_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "eucl_scene_parse": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "eucl_parsed_texture_count": (C.c_int, [C.c_void_p]),
    "eucl_parsed_texture_path": (C.c_char_p, [C.c_void_p, C.c_int]),
    "eucl_parsed_set_texture": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p]),
    "eucl_parsed_flat": (C.POINTER(EuclFlatScene), [C.c_void_p]),
    "eucl_parsed_destroy": (None, [C.c_void_p]),
    "eucl_device_count": (C.c_int, []),
    "eucl_last_error": (C.c_char_p, []),
    "eucl_version": (C.c_char_p, []),
    "eucl_scene_create": (C.c_int, [C.POINTER(EuclFlatScene), C.c_int, C.POINTER(C.c_void_p)]),
    "eucl_scene_create_precision": (C.c_int, [C.POINTER(EuclFlatScene), C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "eucl_scene_destroy": (None, [C.c_void_p]),
    "eucl_scene_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "eucl_band_rows_for_rank": (C.c_uint32, [C.POINTER(EuclRenderOpts)]),
    "eucl_render": (C.c_int, [C.c_void_p, C.POINTER(EuclCamera), C.POINTER(EuclRenderOpts), C.c_void_p, C.c_void_p,
                              C.POINTER(EuclStats)]),
    "eucl_render_device": (C.c_int, [C.c_void_p, C.POINTER(EuclCamera), C.POINTER(EuclRenderOpts), C.c_void_p,
                                     C.c_void_p, C.POINTER(EuclStats)]),
    "eucl_render_frames": (C.c_int, [C.c_void_p, C.POINTER(EuclFrame), C.c_uint32, C.POINTER(EuclRenderOpts), C.c_void_p,
                                     C.c_void_p, C.POINTER(EuclStats)]),
    "eucl_render_frames_device": (C.c_int, [C.c_void_p, C.POINTER(EuclFrame), C.c_uint32, C.POINTER(EuclRenderOpts),
                                            C.c_void_p, C.c_void_p, C.POINTER(EuclStats)]),
    "eucl_render_aovs": (C.c_int, [C.c_void_p, C.POINTER(EuclFrame), C.c_uint32, C.POINTER(EuclRenderOpts), C.c_void_p,
                                   C.c_void_p, C.POINTER(EuclAovs), C.POINTER(EuclStats)]),
    "eucl_render_aovs_device": (C.c_int, [C.c_void_p, C.POINTER(EuclFrame), C.c_uint32, C.POINTER(EuclRenderOpts),
                                          C.c_void_p, C.c_void_p, C.POINTER(EuclAovs), C.POINTER(EuclStats)]),
    "eucl_trace_rays": (C.c_int, [C.c_void_p, C.POINTER(EuclRays), C.c_void_p, C.c_void_p, C.POINTER(EuclAovs),
                                  C.POINTER(EuclStats)]),
    "eucl_trace_rays_device": (C.c_int, [C.c_void_p, C.POINTER(EuclRays), C.c_void_p, C.c_void_p, C.POINTER(EuclAovs),
                                         C.POINTER(EuclStats)]),
    "eucl_render_trees": (C.c_int, [C.c_void_p, C.POINTER(EuclFrame), C.c_uint32, C.POINTER(EuclRenderOpts), C.c_void_p,
                                    C.c_void_p, C.POINTER(EuclTreeQuery), C.POINTER(EuclStats)]),
    "eucl_trace_ray_trees": (C.c_int, [C.c_void_p, C.POINTER(EuclRays), C.c_void_p, C.c_void_p, C.POINTER(EuclTreeQuery),
                                       C.POINTER(EuclStats)]),
    "eucl_trace_path": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double,
                                  C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "eucl_locate_points": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "eucl_locate_points_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "eucl_trace_paths": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                   C.c_void_p, C.c_void_p]),
    "eucl_trace_paths_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "eucl_camera_rotate_yaw": (C.c_int, [C.POINTER(EuclCamera), C.c_double, C.c_int]),
    "eucl_camera_rotate_pitch": (C.c_int, [C.POINTER(EuclCamera), C.c_double, C.c_int]),
    "eucl_camera_rotate_roll": (C.c_int, [C.POINTER(EuclCamera), C.c_double]),
    "eucl_camera_rotate_plane4": (C.c_int, [C.POINTER(EuclCamera), C.c_int, C.c_int, C.c_double]),
    "eucl_device_malloc": (C.c_int, [C.c_int, C.c_uint64, C.POINTER(C.c_void_p)]),
    "eucl_device_free": (C.c_int, [C.c_int, C.c_void_p]),
    "eucl_scene_memory": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "eucl_host_register": (C.c_int, [C.c_void_p, C.c_uint64]),
    "eucl_host_unregister": (C.c_int, [C.c_void_p]),
    "eucl_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "eucl_ipc_open": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "eucl_ipc_close": (C.c_int, [C.c_void_p]),
    "eucl_write_ppm": (C.c_int, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_void_p]),
    "eucl_fp64_peak": (C.c_int, [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

import os as _os

LIB_PATH = Path(__file__).resolve().parent / f"libeuclider_b200{_os.environ.get('EUCL_LIB_SUFFIX', '')}.so"
_lib = None


class EuclError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"{STATUS_NAMES.get(status, status)}: {message}")
        self.status = status
        self.message = message


def lib() -> C.CDLL:
    """Loads libeuclider_b200.so (built in-tree by euclider_b200._build / __graft_entry__.build)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(there is no CPU fallback)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (restype, argtypes) in PROTOTYPES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export it
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != EUCL_OK:
        raise EuclError(status, lib().eucl_last_error().decode("utf-8", "replace"))
