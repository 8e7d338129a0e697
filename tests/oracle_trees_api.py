"""ctypes binding of the ray-tree oracle (tests/oracle_trees.cc): the CPU oracle of oracle/oracle.cc, unchanged, plus
oracle_ray_tree, which defines the trees of eucl_render_trees / eucl_trace_ray_trees bit for bit, and first_difference,
which names the first node and field in which two trees differ.

Test infrastructure: imported only by tests/ and __graft_entry__.build().
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path
from typing import Optional, Sequence

import numpy as np

import oracle_rays_api
from euclider_b200 import TREE_NODE_DTYPE, RayTree
from euclider_b200._capi import EUCL_MAX_LEVELS, EuclFlatScene

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"

# the det build (deterministic libm, bit-comparable with the f64 kernels) and the f32 build (`low_precision`)
TREES_SOURCE = ROOT / "tests" / "oracle_trees.cc"
TREES_FLAGS = {"det": ["-DORACLE_DETMATH"], "f32": ["-DORACLE_DETMATH", "-DORACLE_F32"]}
_libs = {}


def trees_lib_path(variant: str) -> Path:
    return ROOT / "build" / f"liboracle_trees_{variant}.so"


def build_trees(variant: str) -> Path:
    """Compiles the tree oracle with the flags of oracle/Makefile."""
    path = trees_lib_path(variant)
    path.parent.mkdir(exist_ok=True)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra",
           "-pthread", *TREES_FLAGS[variant], "-I", str(ROOT / "include"), "-shared", "-o", str(path), str(TREES_SOURCE)]
    subprocess.run(cmd, check=True, capture_output=True)
    return path


def trees_lib(variant: str = "det") -> C.CDLL:
    if variant not in _libs:
        path = trees_lib_path(variant)
        deps = [TREES_SOURCE, ORACLE_DIR / "oracle.cc", ROOT / "include" / "euclider_b200.h", ROOT / "include" / "eucl_detmath.h"]
        if not path.exists() or path.stat().st_mtime < max(d.stat().st_mtime for d in deps):
            build_trees(variant)
        h = C.CDLL(str(path))
        h.oracle_ray_tree.restype = C.c_int
        h.oracle_ray_tree.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_uint32, C.c_double,
                                      C.c_uint32, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p]
        h.oracle_tree_pixel.restype = None
        h.oracle_tree_pixel.argtypes = [C.c_void_p, C.c_void_p]
        _libs[variant] = h
    return _libs[variant]


def variant_of(env) -> str:
    return "f32" if env.precision == "f32" else "det"


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
    rc = trees_lib(variant).oracle_ray_tree(C.byref(env.flat), o.ctypes.data, d.ctypes.data, int(cell[0]), int(cell[1]), depth,
                                            float(time), int(capacity), nodes.ctypes.data, C.byref(count), levels.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_ray_tree failed: {rc}")
    tree = RayTree(nodes[:min(count.value, int(capacity))], count.value, env.dim, "f32" if variant == "f32" else "f64")
    return (tree, levels[:depth + 1]) if level_counts else tree


def pixel_trees(env, width: int, height: int, pixels: Sequence, time: float = 0.0, camera=None, capacity: int = 4096,
                variant: Optional[str] = None, level_counts: bool = False):
    """The oracle's trees of camera pixels (x, y) of a width x height frame: the rays of oracle_camera_rays."""
    variant = variant or variant_of(env)
    origins, directions = oracle_rays_api.camera_rays(env, width, height, camera=camera, variant=variant)
    cam = camera if camera is not None else env.camera
    return [ray_tree(env, origins[y, x], directions[y, x], (x, y), int(cam.max_depth), time, capacity, variant, level_counts)
            for x, y in pixels]


def tree_pixel(root, variant: str = "det") -> np.ndarray:
    """RGB8 of a tree's root: composited over opaque white and quantised (a checkerboard root as it is)."""
    rec = np.ascontiguousarray(np.asarray(root, dtype=TREE_NODE_DTYPE).reshape(1))
    out = np.zeros(3, np.uint8)
    trees_lib(variant).oracle_tree_pixel(rec.ctypes.data, out.ctypes.data)
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
