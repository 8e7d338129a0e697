"""ctypes binding of the AOV oracle (tests/oracle_aovs.cc): the CPU oracle of oracle/oracle.cc, unchanged, plus
oracle_render_aovs, which defines the per-pixel auxiliary outputs bit for bit.

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
AOV_SOURCE = ROOT / "tests" / "oracle_aovs.cc"
AOV_FLAGS = {"det": ["-DORACLE_DETMATH"], "f32": ["-DORACLE_DETMATH", "-DORACLE_F32"]}
_aov_libs = {}


def aov_lib_path(variant: str) -> Path:
    return ROOT / "build" / f"liboracle_aovs_{variant}.so"


def build_aovs(variant: str) -> Path:
    """Compiles the AOV oracle with the flags of oracle/Makefile."""
    path = aov_lib_path(variant)
    path.parent.mkdir(exist_ok=True)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra",
           "-pthread", *AOV_FLAGS[variant], "-I", str(ROOT / "include"), "-shared", "-o", str(path), str(AOV_SOURCE)]
    subprocess.run(cmd, check=True, capture_output=True)
    return path


def aov_lib(variant: str = "det") -> C.CDLL:
    if variant not in _aov_libs:
        path = aov_lib_path(variant)
        deps = [AOV_SOURCE, ORACLE_DIR / "oracle.cc", ROOT / "include" / "euclider_b200.h", ROOT / "include" / "eucl_detmath.h"]
        if not path.exists() or path.stat().st_mtime < max(d.stat().st_mtime for d in deps):
            build_aovs(variant)
        h = C.CDLL(str(path))
        h.oracle_render_aovs.restype = C.c_int
        h.oracle_render_aovs.argtypes = [C.POINTER(EuclFlatScene), C.POINTER(EuclCamera), C.c_uint32, C.c_uint32, C.c_double,
                                         C.c_uint32, C.c_uint32, C.c_int] + [C.c_void_p] * 8
        _aov_libs[variant] = h
    return _aov_libs[variant]


def render_aovs(env, width: int, height: int, time: float = 0.0, threads: int | None = None, rows=None, camera=None,
                variant: str = "det"):
    """Oracle frame with every AOV plane: (rgb, hit, aovs dict, stats dict).  aovs: depth float32 [rows,w], position and
    normal float32 [rows,w,dim], segments and levels uint32 [rows,w] -- include/euclider_b200.h, EuclAovs."""
    threads = threads or os.cpu_count() or 1
    r0, r1 = rows if rows is not None else (0, height)
    n, dim = r1 - r0, env.dim
    rgb = np.zeros((n, width, 3), dtype=np.uint8)
    hit = np.zeros((n, width), dtype=np.int32)
    aovs = {"depth": np.zeros((n, width), np.float32), "position": np.zeros((n, width, dim), np.float32),
            "normal": np.zeros((n, width, dim), np.float32), "segments": np.zeros((n, width), np.uint32),
            "levels": np.zeros((n, width), np.uint32)}
    stats = np.zeros(8 + EUCL_MAX_LEVELS, dtype=np.uint64)
    cam = camera if camera is not None else env.camera
    flat = env.flat
    rc = aov_lib(variant).oracle_render_aovs(C.byref(flat), C.byref(cam), width, height, float(time), r0, r1, threads,
                                             rgb.ctypes.data, hit.ctypes.data, *(a.ctypes.data for a in aovs.values()),
                                             stats.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_render_aovs failed: {rc}")
    levels = int(cam.max_depth) + 1
    return rgb, hit, aovs, {"segments": int(stats[0]), "nodes": int(stats[1]),
                            "level_counts": [int(v) for v in stats[8:8 + levels]]}
