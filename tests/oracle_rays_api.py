"""ctypes binding of the ray oracle (tests/oracle_rays.cc): the CPU oracle of oracle/oracle.cc, unchanged, plus
oracle_trace_rays, which defines eucl_trace_rays bit for bit, and oracle_camera_rays, the camera's own rays.

Test infrastructure: imported only by tests/ and __graft_entry__.build().
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from euclider_b200._capi import EUCL_MAX_LEVELS, EuclCamera, EuclFlatScene

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"

# the det build (deterministic libm, bit-comparable with the f64 kernels) and the f32 build (`low_precision`)
RAYS_SOURCE = ROOT / "tests" / "oracle_rays.cc"
RAYS_FLAGS = {"det": ["-DORACLE_DETMATH"], "f32": ["-DORACLE_DETMATH", "-DORACLE_F32"]}
_libs = {}


def rays_lib_path(variant: str) -> Path:
    return ROOT / "build" / f"liboracle_rays_{variant}.so"


def build_rays(variant: str) -> Path:
    """Compiles the ray oracle with the flags of oracle/Makefile."""
    path = rays_lib_path(variant)
    path.parent.mkdir(exist_ok=True)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra",
           "-pthread", *RAYS_FLAGS[variant], "-I", str(ROOT / "include"), "-shared", "-o", str(path), str(RAYS_SOURCE)]
    subprocess.run(cmd, check=True, capture_output=True)
    return path


def rays_lib(variant: str = "det") -> C.CDLL:
    if variant not in _libs:
        path = rays_lib_path(variant)
        deps = [RAYS_SOURCE, ORACLE_DIR / "oracle.cc", ROOT / "include" / "euclider_b200.h", ROOT / "include" / "eucl_detmath.h"]
        if not path.exists() or path.stat().st_mtime < max(d.stat().st_mtime for d in deps):
            build_rays(variant)
        h = C.CDLL(str(path))
        h.oracle_trace_rays.restype = C.c_int
        h.oracle_trace_rays.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                        C.c_double, C.c_int] + [C.c_void_p] * 8
        h.oracle_camera_rays.restype = C.c_int
        h.oracle_camera_rays.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p]
        _libs[variant] = h
    return _libs[variant]


def camera_rays(env, width: int, height: int, camera=None, variant: str = "det"):
    """(origins, directions) of the camera's width x height rays, float64 (height, width, dim), row 0 = bottom."""
    cam = camera if camera is not None else env.camera
    origins = np.zeros((height, width, env.dim), np.float64)
    directions = np.zeros_like(origins)
    rc = rays_lib(variant).oracle_camera_rays(C.byref(env.flat), C.byref(cam), width, height, origins.ctypes.data,
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
    lead, dim = o.shape[:-1], env.dim
    n = int(np.prod(lead, dtype=np.int64))
    if width is None:
        width = lead[-1] if len(lead) >= 2 else 1
    depth = int(env.camera.max_depth) if max_depth is None else int(max_depth)
    rgb = np.zeros(lead + (3,), dtype=np.uint8)
    hit = np.zeros(lead, dtype=np.int32)
    aovs = {"depth": np.zeros(lead, np.float32), "position": np.zeros(lead + (dim,), np.float32),
            "normal": np.zeros(lead + (dim,), np.float32), "segments": np.zeros(lead, np.uint32),
            "levels": np.zeros(lead, np.uint32)}
    stats = np.zeros(8 + EUCL_MAX_LEVELS, dtype=np.uint64)
    rc = rays_lib(variant).oracle_trace_rays(C.byref(env.flat), o.ctypes.data, d.ctypes.data, n, int(width), depth,
                                             float(time), threads, rgb.ctypes.data, hit.ctypes.data,
                                             *(a.ctypes.data for a in aovs.values()), stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_trace_rays failed: {rc}")
    return rgb, hit, aovs, {"segments": int(stats[0]), "nodes": int(stats[1]),
                            "level_counts": [int(v) for v in stats[8:8 + depth + 1]]}
