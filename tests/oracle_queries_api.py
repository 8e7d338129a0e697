"""ctypes binding of the query oracle (tests/oracle_queries.cc): the CPU oracle of oracle/oracle.cc, unchanged, plus
oracle_locate, Universe::material_at for many points, in the f64 `det` build and the f32 build.

Test infrastructure: imported only by tests/ and __graft_entry__.build().
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from euclider_b200._capi import EuclFlatScene

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"

QUERIES_SOURCE = ROOT / "tests" / "oracle_queries.cc"
QUERIES_FLAGS = {"det": ["-DORACLE_DETMATH"], "f32": ["-DORACLE_DETMATH", "-DORACLE_F32"]}
_libs = {}


def queries_lib_path(variant: str) -> Path:
    return ROOT / "build" / f"liboracle_queries_{variant}.so"


def build_queries(variant: str) -> Path:
    """Compiles the query oracle with the flags of oracle/Makefile."""
    path = queries_lib_path(variant)
    path.parent.mkdir(exist_ok=True)
    cmd = [os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-Wall", "-Wextra",
           "-pthread", *QUERIES_FLAGS[variant], "-I", str(ROOT / "include"), "-shared", "-o", str(path), str(QUERIES_SOURCE)]
    subprocess.run(cmd, check=True, capture_output=True)
    return path


def queries_lib(variant: str = "det") -> C.CDLL:
    if variant not in _libs:
        path = queries_lib_path(variant)
        deps = [QUERIES_SOURCE, ORACLE_DIR / "oracle.cc", ROOT / "include" / "euclider_b200.h", ROOT / "include" / "eucl_detmath.h"]
        if not path.exists() or path.stat().st_mtime < max(d.stat().st_mtime for d in deps):
            build_queries(variant)
        h = C.CDLL(str(path))
        h.oracle_locate.restype = C.c_int
        h.oracle_locate.argtypes = [C.POINTER(EuclFlatScene), C.c_void_p, C.c_uint32, C.c_void_p]
        _libs[variant] = h
    return _libs[variant]


def locate(env, points, variant: str = "det") -> np.ndarray:
    """Oracle of Environment.locate: int32 of the points' leading shape."""
    p = np.ascontiguousarray(points, dtype=np.float64)
    assert p.shape[-1] == env.dim
    out = np.zeros(p.shape[:-1], np.int32)
    rc = queries_lib(variant).oracle_locate(C.byref(env.flat), p.ctypes.data, out.size, out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"oracle_locate failed: {rc}")
    return out
