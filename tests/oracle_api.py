"""ctypes binding of the CPU oracle -- the restatement used as the parity checker: oracle/liboracle*.so (oracle.cc: frames,
paths and the unit-test hooks) and oracle/liboracle_features_{det,f32}.so (oracle_features.cc: AOV planes, caller rays,
ray trees and universe queries).  Every library is built by oracle/Makefile, which decides when one is stale.

Test infrastructure: imported only by tests/, tools/, __graft_entry__.smoke() and bench.py's CPU legs.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path
from typing import Optional, Sequence

import numpy as np

from euclider_b200 import TREE_NODE_DTYPE, RayTree
from euclider_b200._capi import EUCL_MAX_LEVELS, EuclCamera, EuclFlatScene, EuclPrim

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
LIB_PATHS = {"glibc": ORACLE_DIR / "liboracle.so", "det": ORACLE_DIR / "liboracle_det.so",
             "count": ORACLE_DIR / "liboracle_count.so",  # "count": det + flop counters (tools/oracle_flops.py)
             "f32": ORACLE_DIR / "liboracle_f32.so"}  # the reference's `low_precision` feature (type F = f32), det libm
# the feature statements over the det build (bit-comparable with the f64 kernels) and the f32 build
FEATURE_PATHS = {"det": ORACLE_DIR / "liboracle_features_det.so", "f32": ORACLE_DIR / "liboracle_features_f32.so"}
_libs = {}
_features = {}

dptr = C.POINTER(C.c_double)


def build(target: str = "all") -> None:
    subprocess.run(["make", "-C", str(ORACLE_DIR), target], check=True, capture_output=True)


def lib(variant: str = "det") -> C.CDLL:
    """variant "det": transcendental functions from include/eucl_detmath.h (bit-comparable with the
    CUDA path); "glibc": the host libm (what the Rust reference would link on this platform); "f32": the `det` build
    with `type F = f32` (renderer and camera path only: the unit-test hooks probe the f64 builds)."""
    if variant not in _libs:
        path = LIB_PATHS[variant]
        build(path.name)
        h = C.CDLL(str(path))
        h.oracle_render.restype = C.c_int
        h.oracle_render.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_uint32, C.c_uint32, C.c_double,
                                    C.c_uint32, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        if variant != "f32":
            h.oracle_entity_intersections.restype = C.c_int
            h.oracle_entity_intersections.argtypes = [C.POINTER(EuclFlatScene), C.c_int, dptr, dptr, C.c_int, dptr]
            h.oracle_prim_intersect.restype = C.c_int
            h.oracle_prim_intersect.argtypes = [C.c_int, C.POINTER(EuclPrim), dptr, dptr, dptr]
            h.oracle_prim_inside.restype = C.c_int
            h.oracle_prim_inside.argtypes = [C.c_int, C.POINTER(EuclPrim), dptr]
            h.oracle_entity_inside.restype = C.c_int
            h.oracle_entity_inside.argtypes = [C.POINTER(EuclFlatScene), C.c_int, dptr]
            h.oracle_material_at.restype = C.c_int
            h.oracle_material_at.argtypes = [C.POINTER(EuclFlatScene), dptr]
            h.oracle_angle_between.restype = C.c_double
            h.oracle_angle_between.argtypes = [C.c_int, dptr, dptr]
            h.oracle_angle_between_f32.restype = C.c_float
            h.oracle_angle_between_f32.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float)]
            h.oracle_combine_palette_color.restype = None
            h.oracle_combine_palette_color.argtypes = [dptr, dptr, C.c_double, dptr]
            h.oracle_combine_palette_color_f32.restype = None
            h.oracle_combine_palette_color_f32.argtypes = [C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_float,
                                                           C.POINTER(C.c_float)]
            h.oracle_remainder_i.restype = C.c_int64
            h.oracle_remainder_i.argtypes = [C.c_int64, C.c_int64]
            h.oracle_remainder_f.restype = C.c_double
            h.oracle_remainder_f.argtypes = [C.c_double, C.c_double]
            h.oracle_blend.restype = None
            h.oracle_blend.argtypes = [C.c_int, C.c_double, dptr, dptr, dptr]
            h.oracle_to_pixel.restype = None
            h.oracle_to_pixel.argtypes = [dptr, C.POINTER(C.c_uint8)]
            h.oracle_perlin4.restype = C.c_double
            h.oracle_perlin4.argtypes = [C.POINTER(C.c_uint8), dptr]
            h.oracle_hsv_to_rgb.restype = None
            h.oracle_hsv_to_rgb.argtypes = [C.c_double, C.c_double, C.c_double, dptr]
            h.oracle_general_rotation.restype = None
            h.oracle_general_rotation.argtypes = [C.c_int, dptr, dptr, C.c_double, dptr, dptr]
            h.oracle_surface_probe.restype = None
            h.oracle_surface_probe.argtypes = [C.POINTER(EuclFlatScene), C.c_int, dptr, dptr, C.c_int, dptr, dptr, dptr]
            h.oracle_mapped_color.restype = None
            h.oracle_mapped_color.argtypes = [C.POINTER(EuclFlatScene), C.c_int, dptr, dptr]
            h.oracle_ray_vector.restype = None
            h.oracle_ray_vector.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_int, C.c_int, C.c_int,
                                            C.c_int, dptr]
            h.oracle_detmath_unary.restype = None
            h.oracle_detmath_unary.argtypes = [C.c_int, dptr, dptr, C.c_int]
            h.oracle_detmath_atan2.restype = None
            h.oracle_detmath_atan2.argtypes = [dptr, dptr, dptr, C.c_int]
        h.oracle_trace_path.restype = C.c_int
        h.oracle_trace_path.argtypes = [C.POINTER(EuclFlatScene), dptr, dptr, C.c_double, dptr, dptr]
        h.oracle_uses_detmath.restype = C.c_int
        h.oracle_real_bytes.restype = C.c_int
        _libs[variant] = h
    return _libs[variant]


def darr(values):
    values = list(values)
    return (C.c_double * len(values))(*values)


def render(env, width: int, height: int, time: float = 0.0, threads: int | None = None, rows=None, camera=None,
           variant: str = "det"):
    """Oracle frame for an euclider_b200.Environment: (rgb uint8 [rows,w,3], hit int32 [rows,w], stats dict)."""
    threads = threads or os.cpu_count() or 1
    r0, r1 = rows if rows is not None else (0, height)
    rgb = np.zeros((r1 - r0, width, 3), dtype=np.uint8)
    hit = np.zeros((r1 - r0, width), dtype=np.int32)
    stats = np.zeros(8 + EUCL_MAX_LEVELS, dtype=np.uint64)
    cam = camera if camera is not None else env.camera
    flat = env.flat
    rc = lib(variant).oracle_render(C.byref(flat), C.byref(cam), width, height, float(time), r0, r1, threads,
                             rgb.ctypes.data, hit.ctypes.data, stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_render failed: {rc}")
    levels = int(cam.max_depth) + 1
    return rgb, hit, {
        "segments": int(stats[0]), "nodes": int(stats[1]), "nan_channel": int(stats[2]), "bad_texcoord": int(stats[3]),
        "no_material": int(stats[4]), "csg_runaway": int(stats[5]), "flops": int(stats[6]),
        "level_counts": [int(v) for v in stats[8:8 + levels]],
    }


def trace_path(env, location, direction, distance: float, variant: str = "det"):
    """Universe::trace_path_unknown on the oracle: (location, direction) or None."""
    dim = env.dim
    out_l, out_d = (C.c_double * dim)(), (C.c_double * dim)()
    flat = env.flat
    rc = lib(variant).oracle_trace_path(C.byref(flat), darr(location), darr(direction), float(distance), out_l, out_d)
    if rc == 1:
        return None
    if rc != 0:
        raise RuntimeError("oracle_trace_path: runaway")
    return list(out_l), list(out_d)


def features(variant: str = "det") -> C.CDLL:
    """The feature statements of oracle/oracle_features.cc over the "det" or the "f32" build of the oracle."""
    if variant not in _features:
        path = FEATURE_PATHS[variant]
        build(path.name)
        h = C.CDLL(str(path))
        h.oracle_render_aovs.restype = C.c_int
        h.oracle_render_aovs.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_uint32, C.c_uint32, C.c_double,
                                         C.c_uint32, C.c_uint32, C.c_int] + [C.c_void_p] * 8
        h.oracle_trace_rays.restype = C.c_int
        h.oracle_trace_rays.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                        C.c_double, C.c_int] + [C.c_void_p] * 8
        h.oracle_camera_rays.restype = C.c_int
        h.oracle_camera_rays.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p]
        h.oracle_ray_tree.restype = C.c_int
        h.oracle_ray_tree.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_double,
                                      C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]
        h.oracle_tree_pixel.restype = None
        h.oracle_tree_pixel.argtypes = [C.c_void_p, C.c_void_p]
        h.oracle_locate.restype = C.c_int
        h.oracle_locate.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_uint32, C.c_void_p]
        _features[variant] = h
    return _features[variant]


def variant_of(env) -> str:
    return "f32" if env.precision == "f32" else "det"


def _aov_planes(lead, dim):
    """Zeroed AOV planes in the argument order of oracle_render_aovs / oracle_trace_rays (include/euclider_b200.h,
    EuclAovs): depth float32, position and normal float32 [..., dim], segments and levels uint32."""
    return {"depth": np.zeros(lead, np.float32), "position": np.zeros(lead + (dim,), np.float32),
            "normal": np.zeros(lead + (dim,), np.float32), "segments": np.zeros(lead, np.uint32),
            "levels": np.zeros(lead, np.uint32)}


def render_aovs(env, width: int, height: int, time: float = 0.0, threads: int | None = None, rows=None, camera=None,
                variant: str = "det"):
    """Oracle frame with every AOV plane: (rgb, hit, aovs dict, stats dict).  aovs: depth float32 [rows,w], position and
    normal float32 [rows,w,dim], segments and levels uint32 [rows,w] -- include/euclider_b200.h, EuclAovs."""
    threads = threads or os.cpu_count() or 1
    r0, r1 = rows if rows is not None else (0, height)
    n = r1 - r0
    rgb = np.zeros((n, width, 3), dtype=np.uint8)
    hit = np.zeros((n, width), dtype=np.int32)
    aovs = _aov_planes((n, width), env.dim)
    stats = np.zeros(8 + EUCL_MAX_LEVELS, dtype=np.uint64)
    cam = camera if camera is not None else env.camera
    flat = env.flat
    rc = features(variant).oracle_render_aovs(C.byref(flat), C.byref(cam), width, height, float(time), r0, r1, threads,
                                              rgb.ctypes.data, hit.ctypes.data, *(a.ctypes.data for a in aovs.values()),
                                              stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_render_aovs failed: {rc}")
    levels = int(cam.max_depth) + 1
    return rgb, hit, aovs, {"segments": int(stats[0]), "nodes": int(stats[1]),
                            "level_counts": [int(v) for v in stats[8:8 + levels]]}


def camera_rays(env, width: int, height: int, camera=None, variant: str = "det"):
    """(origins, directions) of the camera's width x height rays, float64 (height, width, dim), row 0 = bottom."""
    cam = camera if camera is not None else env.camera
    origins = np.zeros((height, width, env.dim), np.float64)
    directions = np.zeros_like(origins)
    rc = features(variant).oracle_camera_rays(C.byref(env.flat), C.byref(cam), width, height, origins.ctypes.data,
                                              directions.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_camera_rays failed: {rc}")
    return origins, directions


def trace_rays(env, origins, directions, time: float = 0.0, max_depth: int | None = None, width: int | None = None,
               threads: int | None = None, variant: str = "det"):
    """Oracle of Environment.trace_rays with every AOV plane: (rgb, hit, aovs dict, stats dict), leading shape of the rays.
    `width` defaults as in Environment.trace_rays."""
    threads = threads or os.cpu_count() or 1
    o = np.ascontiguousarray(origins, dtype=np.float64)
    d = np.ascontiguousarray(directions, dtype=np.float64)
    assert o.shape == d.shape and o.shape[-1] == env.dim
    lead = o.shape[:-1]
    n = int(np.prod(lead, dtype=np.int64))
    if width is None:
        width = lead[-1] if len(lead) >= 2 else 1
    depth = int(env.camera.max_depth) if max_depth is None else int(max_depth)
    rgb = np.zeros(lead + (3,), dtype=np.uint8)
    hit = np.zeros(lead, dtype=np.int32)
    aovs = _aov_planes(lead, env.dim)
    stats = np.zeros(8 + EUCL_MAX_LEVELS, dtype=np.uint64)
    rc = features(variant).oracle_trace_rays(C.byref(env.flat), o.ctypes.data, d.ctypes.data, n, int(width), depth,
                                             float(time), threads, rgb.ctypes.data, hit.ctypes.data,
                                             *(a.ctypes.data for a in aovs.values()), stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_trace_rays failed: {rc}")
    return rgb, hit, aovs, {"segments": int(stats[0]), "nodes": int(stats[1]),
                            "level_counts": [int(v) for v in stats[8:8 + depth + 1]]}


def ray_tree(env, origin, direction, cell=(0, 0), max_depth: Optional[int] = None, time: float = 0.0, capacity: int = 4096,
             variant: Optional[str] = None, level_counts: bool = False):
    """The oracle's tree of one item with ray (origin, direction) and grid cell `cell` (its checkerboard when the origin lies
    in no entity): a RayTree, and with level_counts=True also the per-level trace calls."""
    variant = variant or variant_of(env)
    depth = int(env.camera.max_depth) if max_depth is None else int(max_depth)
    o = np.ascontiguousarray(origin, dtype=np.float64)
    d = np.ascontiguousarray(direction, dtype=np.float64)
    nodes = np.zeros(max(int(capacity), 1), TREE_NODE_DTYPE)
    count = C.c_uint32()
    levels = np.zeros(EUCL_MAX_LEVELS, np.uint64)
    rc = features(variant).oracle_ray_tree(C.byref(env.flat), o.ctypes.data, d.ctypes.data, int(cell[0]), int(cell[1]), depth,
                                           float(time), int(capacity), nodes.ctypes.data, C.byref(count), levels.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_ray_tree failed: {rc}")
    tree = RayTree(nodes[:min(count.value, int(capacity))], count.value, env.dim, "f32" if variant == "f32" else "f64")
    return (tree, levels[:depth + 1]) if level_counts else tree


def pixel_trees(env, width: int, height: int, pixels: Sequence, time: float = 0.0, camera=None, capacity: int = 4096,
                variant: Optional[str] = None, level_counts: bool = False):
    """The oracle's trees of camera pixels (x, y) of a width x height frame: the rays of oracle_camera_rays."""
    variant = variant or variant_of(env)
    origins, directions = camera_rays(env, width, height, camera=camera, variant=variant)
    cam = camera if camera is not None else env.camera
    return [ray_tree(env, origins[y, x], directions[y, x], (x, y), int(cam.max_depth), time, capacity, variant, level_counts)
            for x, y in pixels]


def tree_pixel(root, variant: str = "det") -> np.ndarray:
    """RGB8 of a tree's root: composited over opaque white and quantised (a checkerboard root as it is)."""
    rec = np.ascontiguousarray(np.asarray(root, dtype=TREE_NODE_DTYPE).reshape(1))
    out = np.zeros(3, np.uint8)
    features(variant).oracle_tree_pixel(rec.ctypes.data, out.ctypes.data)
    return out


def _bits(v) -> str:
    return f"{np.float64(v).view(np.uint64):#018x}"


def first_difference(a: RayTree, b: RayTree) -> Optional[str]:
    """None when the two trees are equal bit for bit (any NaN equals any NaN) with equal counts; else the first node and
    field that differ, e.g. "node 5, level 3, reflected: t 0x... vs 0x..." (floats as their bit patterns)."""
    kinds = ("root", "transmitted", "reflected")
    for j in range(min(len(a.nodes), len(b.nodes))):
        x, y = a.nodes[j], b.nodes[j]
        where = f"node {j}, level {int(x['level'])}, {kinds[int(x['kind'])] if 0 <= x['kind'] < 3 else x['kind']}"
        for name in TREE_NODE_DTYPE.names:
            u, v = np.atleast_1d(x[name]), np.atleast_1d(y[name])
            if u.dtype.kind == "f":
                same = (u.view(np.uint64) == v.view(np.uint64)) | (np.isnan(u) & np.isnan(v))
                if not same.all():
                    k = int(np.flatnonzero(~same)[0])
                    comp = f"[{k}]" if len(u) > 1 else ""
                    return f"{where}: {name}{comp} {_bits(u[k])} vs {_bits(v[k])} ({u[k]!r} vs {v[k]!r})"
            elif not np.array_equal(u, v):
                return f"{where}: {name} {u.tolist() if len(u) > 1 else int(u[0])} vs {v.tolist() if len(v) > 1 else int(v[0])}"
    if a.count != b.count or len(a.nodes) != len(b.nodes):
        return f"node count {a.count} vs {b.count} (stored {len(a.nodes)} vs {len(b.nodes)})"
    return None


def locate(env, points, variant: str = "det") -> np.ndarray:
    """Oracle of Environment.locate: int32 of the points' leading shape."""
    p = np.ascontiguousarray(points, dtype=np.float64)
    assert p.shape[-1] == env.dim
    out = np.zeros(p.shape[:-1], np.int32)
    rc = features(variant).oracle_locate(C.byref(env.flat), p.ctypes.data, out.size, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_locate failed: {rc}")
    return out
