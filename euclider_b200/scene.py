"""Host-side mirror of the reference interface for the trace-loop path.

Reference (Rust): ``scene::Parser::default().parse::<Box<Environment>>(json)`` (src/scene.rs:564,
1466-1478) builds an ``Environment``; ``Environment::render(dimensions, time, threads, context)``
(src/universe/mod.rs:300-357) renders one frame into a ``RawImage2d<u8>`` (RGB8, row 0 = bottom).
The same names and argument meanings are kept here; the work is done by libeuclider_b200.so
(C ABI in include/euclider_b200.h) on a B200.  There is no CPU rendering path in this package.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field
from pathlib import Path
from typing import Dict, List, Mapping, Optional, Sequence, Tuple, Union

import numpy as np

from . import _capi
from ._capi import (EuclAovs, EuclCamera, EuclError, EuclFlatScene, EuclFrame, EuclRays, EuclRenderOpts, EuclStats,
                    EuclTreeQuery, EUCL_PIPELINE_MEGAKERNEL, EUCL_PIPELINE_WAVEFRONT, check, lib)

ParserError = EuclError  # the reference's `ParserError` (src/scene.rs:524-552); see EuclError.status

# `resources/universe_dim.jpg` (background of 3d_room / 3d_hallways) is absent from the reference
# checkout (.MISSING_LARGE_BLOBS); the declared substitute is used by the library and the oracle alike.
DEFAULT_TEXTURE_SUBSTITUTES = {"universe_dim.jpg": "universe_bright.jpg", "moon.jpg": "universe_bright.jpg"}


@dataclass
class SimulationContext:
    """The fields of the reference's SimulationContext that `render` reads (src/simulation.rs:167-186)."""
    resolution: int = 1  # the reference defaults to 8 (window / 8); headless renders use 1
    debugging: bool = False


@dataclass
class RawImage2d:
    """glium's RawImage2d<u8> as returned by Environment::render: RGB8, row 0 = bottom."""
    data: np.ndarray  # uint8, shape (height, width, 3)
    width: int
    height: int
    format: str = "U8U8U8"
    hit_ids: Optional[np.ndarray] = None  # int32 (height, width): primary hit entity, -1 background, -2 checkerboard
    stats: Optional[dict] = None
    aovs: Optional[Dict[str, np.ndarray]] = None  # requested AOV planes by name (AOV_NAMES), rows as `data`
    trees: Optional[List["RayTree"]] = None  # requested ray trees, in request order

    def to_top_down(self) -> np.ndarray:
        return self.data[::-1]

    def save(self, path: Union[str, os.PathLike]) -> None:
        """Writes the frame top-down: `.ppm` through the library (eucl_write_ppm), anything else via Pillow."""
        path = str(path)
        if path.lower().endswith(".ppm"):
            check(lib().eucl_write_ppm(path.encode(), self.width, self.height, np.ascontiguousarray(self.data).ctypes.data))
        else:
            from PIL import Image

            Image.fromarray(np.ascontiguousarray(self.to_top_down())).save(path)


@dataclass
class RawFrames:
    """The frames of one Environment.render_frames call: frame k is data[k], RGB8, row 0 = bottom."""
    data: np.ndarray  # uint8, shape (K, height, width, 3)
    width: int
    height: int
    hit_ids: Optional[np.ndarray] = None  # int32 (K, height, width), as RawImage2d.hit_ids
    stats: Optional[dict] = None  # summed over the K frames
    aovs: Optional[Dict[str, np.ndarray]] = None  # requested AOV planes by name, frame k at index k
    trees: Optional[List["RayTree"]] = None  # requested ray trees, in request order

    def __len__(self) -> int:
        return int(self.data.shape[0])

    def frame(self, k: int) -> RawImage2d:
        """Frame k as a RawImage2d (a view, no copy)."""
        return RawImage2d(self.data[k], self.width, self.height, hit_ids=None if self.hit_ids is None else self.hit_ids[k],
                          aovs=None if self.aovs is None else {name: a[k] for name, a in self.aovs.items()})


@dataclass
class RawRays:
    """The outputs of one Environment.trace_rays call, in ray order with the rays' leading shape."""
    data: np.ndarray  # uint8, shape (..., 3): RGB8 of each ray (the checkerboard of its grid cell when its origin is in no entity)
    hit_ids: Optional[np.ndarray] = None  # int32 (...): primary hit entity, -1 a miss, -2 an origin in no entity
    stats: Optional[dict] = None
    aovs: Optional[Dict[str, np.ndarray]] = None  # requested AOV planes by name, leading shape as `data`
    trees: Optional[List["RayTree"]] = None  # requested ray trees, in request order


def equirect_rays(camera: EuclCamera, width: int, height: int) -> Tuple[np.ndarray, np.ndarray]:
    """Equirectangular (360 x 180 degree) panorama rays of a camera pose for Environment.trace_rays: (origins, directions),
    both float64 of shape (height, width, dim), row 0 at the bottom.  Every origin is the camera location; cell (x, y) looks
    at longitude phi = 2 pi ((x + 0.5) / width - 0.5) and latitude theta = pi ((y + 0.5) / height - 0.5) in the 3-space the
    perspective camera's screen spans: cos(theta) (cos(phi) F - sin(phi) L) + sin(theta) U, with F forward, U up and L
    `left` (4-D) or -normalize(F x U) (3-D).  The centre column looks forward, the first and last columns look back."""
    dim = int(camera.dim)
    if dim not in (3, 4):
        raise ValueError("camera.dim must be 3 or 4")
    if int(width) < 1 or int(height) < 1:
        raise ValueError("width and height must be positive")
    f = np.array(camera.forward[:dim], dtype=np.float64)
    u = np.array(camera.up[:dim], dtype=np.float64)
    if dim == 3:
        c = np.cross(f, u)
        left = -c / np.linalg.norm(c)
    else:
        left = np.array(camera.left[:dim], dtype=np.float64)
    phi = 2.0 * np.pi * ((np.arange(width, dtype=np.float64) + 0.5) / width - 0.5)
    theta = np.pi * ((np.arange(height, dtype=np.float64) + 0.5) / height - 0.5)
    ct, st = np.cos(theta)[:, None, None], np.sin(theta)[:, None, None]
    cp, sp = np.cos(phi)[None, :, None], np.sin(phi)[None, :, None]
    directions = ct * (cp * f - sp * left) + st * u
    origins = np.broadcast_to(np.array(camera.location[:dim], dtype=np.float64), directions.shape).copy()
    return origins, np.ascontiguousarray(directions)


def _ray_arrays(origins, directions, dim: int) -> Tuple[np.ndarray, np.ndarray, Tuple[int, ...]]:
    """float64 C-contiguous copies (when needed) of two (..., dim) arrays of one shape, and their leading shape."""
    o = np.ascontiguousarray(origins, dtype=np.float64)
    d = np.ascontiguousarray(directions, dtype=np.float64)
    if o.shape != d.shape:
        raise ValueError(f"origins {o.shape} and directions {d.shape} must have the same shape")
    if o.ndim < 1 or o.shape[-1] != dim:
        raise ValueError(f"rays must have shape (..., {dim}) for this {dim}-D scene, got {o.shape}")
    lead = o.shape[:-1]
    if int(np.prod(lead, dtype=np.int64)) < 1 or int(np.prod(lead, dtype=np.int64)) > 0x7FFFFFFF:
        raise ValueError("trace_rays needs 1 .. 2^31 - 1 rays")
    return o, d, lead


def _point_array(values, dim: int, what: str) -> Tuple[np.ndarray, Tuple[int, ...]]:
    """A float64 C-contiguous copy (when needed) of a (..., dim) array, and its leading shape."""
    a = np.ascontiguousarray(values, dtype=np.float64)
    if a.ndim < 1 or a.shape[-1] != dim:
        raise ValueError(f"{what} must have shape (..., {dim}) for this {dim}-D scene, got {a.shape}")
    n = int(np.prod(a.shape[:-1], dtype=np.int64))
    if n < 1 or n > 0x7FFFFFFF:
        raise ValueError(f"{what}: 1 .. 2^31 - 1 items")
    return a, a.shape[:-1]


def camera_step(direction: Sequence[float], distance: float, dim: int) -> Optional[Tuple[List[float], float]]:
    """The normalisation of Environment.move_camera: (direction / |direction|, distance * |direction|) as the walk's
    direction and length, or None for a zero direction (the camera does not move)."""
    norm = sum(float(v) * float(v) for v in direction[:dim]) ** 0.5
    if norm == 0.0:
        return None
    return [float(v) / norm for v in direction[:dim]], distance * norm


def _ray_struct(n: int, width: int, max_depth: int, pipeline: int, time: float, profile: bool, origins: int = 0,
                directions: int = 0) -> EuclRays:
    width = max(int(width), 1)
    if n % width:
        raise ValueError(f"width {width} does not divide the {n} rays")
    if int(max_depth) < 0 or int(max_depth) + 1 > _capi.EUCL_MAX_LEVELS:
        raise ValueError(f"max_depth must be 0 .. {_capi.EUCL_MAX_LEVELS - 1}")
    return EuclRays(origins=origins, directions=directions, n=n, width=width, max_depth=int(max_depth), pipeline=pipeline,
                    time_seconds=float(time), profile=int(profile))


# Per-pixel auxiliary outputs (include/euclider_b200.h, EuclAovs): name -> (dtype, one value per pixel or `dim` values).
# depth / position / normal: the primary hit (float32, NaN / +inf where there is none); segments / levels: the cost of the
# pixel's ray tree (uint32).  Host planes the library does not write (other ranks' rows of a band-split render) keep
# their fill: NaN for the float planes, 0xFFFFFFFF for the counts.
AOV_NAMES = ("depth", "position", "normal", "segments", "levels")
_AOV_TYPES = {"depth": (np.float32, False), "position": (np.float32, True), "normal": (np.float32, True),
              "segments": (np.uint32, False), "levels": (np.uint32, False)}


def _aov_names(aovs) -> Tuple[str, ...]:
    """The requested plane names, in AOV_NAMES order; ValueError for an unknown one."""
    names = [aovs] if isinstance(aovs, str) else list(aovs)
    unknown = [n for n in names if n not in _AOV_TYPES]
    if unknown:
        raise ValueError(f"unknown AOV plane(s) {unknown}: choose from {AOV_NAMES}")
    return tuple(n for n in AOV_NAMES if n in names)


def _aov_arrays(aovs, lead: Tuple[int, ...], dim: int) -> Dict[str, np.ndarray]:
    """Host planes for `aovs`: a sequence of names (allocated here) or a mapping name -> array to render into (None:
    allocated).  A given array must have the plane's dtype and shape and be C-contiguous."""
    given = dict(aovs) if isinstance(aovs, Mapping) else {}
    out = {}
    for name in _aov_names(list(aovs)):
        dtype, per_dim = _AOV_TYPES[name]
        shape = lead + ((dim,) if per_dim else ())
        a = given.get(name)
        if a is None:
            a = np.full(shape, np.nan if dtype == np.float32 else 0xFFFFFFFF, dtype=dtype)
        elif not isinstance(a, np.ndarray) or a.dtype != dtype or a.shape != shape or not a.flags["C_CONTIGUOUS"]:
            raise ValueError(f"AOV plane {name!r} must be a C-contiguous {np.dtype(dtype).name} array of shape {shape}")
        out[name] = a
    return out


def _aov_struct(pointers: Mapping[str, int]) -> EuclAovs:
    return EuclAovs(**{name: C.c_void_p(int(ptr)) for name, ptr in pointers.items() if ptr})


def _device_aovs(d_aovs: Mapping[str, int]) -> EuclAovs:
    _aov_names(list(d_aovs))
    if not any(d_aovs.values()):
        raise ValueError("d_aovs names no device plane")
    return _aov_struct(d_aovs)


# Ray-tree nodes (include/euclider_b200.h, EuclTreeNode): the C layout, 176 bytes.
TREE_NODE_DTYPE = np.dtype([("parent", "<i4"), ("level", "<i4"), ("kind", "<i4"), ("medium", "<i4"), ("hit_entity", "<i4"),
                            ("exiting", "<i4"), ("flags", "<u4"), ("surface_rgba8", "<u4"), ("ratio", "<f8"), ("t", "<f8"),
                            ("origin", "<f8", (4,)), ("direction", "<f8", (4,)), ("normal", "<f8", (4,)), ("color", "<f8", (4,))])
TREE_KINDS = ("root", "transmitted", "reflected")
TREE_FLAGS = (("background", _capi.EUCL_TREE_BACKGROUND), ("surface", _capi.EUCL_TREE_SURFACE), ("opaque", _capi.EUCL_TREE_OPAQUE),
              ("no_destination", _capi.EUCL_TREE_NO_DESTINATION), ("undefined", _capi.EUCL_TREE_UNDEFINED),
              ("checkerboard", _capi.EUCL_TREE_CHECKERBOARD))


@dataclass
class RayTree:
    """The ray tree behind one pixel or ray: one node per Universe::trace call, in pre-order (a node, its transmitted
    subtree, its reflected subtree).  Field meanings are those of EuclTreeNode in include/euclider_b200.h."""
    nodes: np.ndarray  # TREE_NODE_DTYPE: the first min(count, capacity) nodes
    count: int         # nodes of the whole tree
    dim: int
    precision: str = "f64"  # the scene's real: every float field holds a value of this type

    @property
    def truncated(self) -> bool:
        return self.count > len(self.nodes)

    def children(self, j: int) -> List[int]:
        """Indices of node j's stored children: the transmitted one first, then the reflected one."""
        return [int(i) for i in np.flatnonzero(self.nodes["parent"] == int(j))]

    def locations(self) -> np.ndarray:
        """Hit locations o + d * t in the scene's precision (the intersectors' expression), (n, dim) float64; NaN where a
        node has no hit."""
        ft = np.float32 if self.precision == "f32" else np.float64
        o = self.nodes["origin"][:, :self.dim].astype(ft)
        d = self.nodes["direction"][:, :self.dim].astype(ft)
        t = self.nodes["t"].astype(ft)[:, None]
        with np.errstate(invalid="ignore", over="ignore"):
            p = (o + d * t).astype(np.float64)
        p[self.nodes["hit_entity"] < 0] = np.nan
        return p

    def format(self) -> str:
        """An indented text view, one line per node."""
        lines = []
        for j, nd in enumerate(self.nodes):
            flags = "|".join(name for name, bit in TREE_FLAGS if int(nd["flags"]) & bit) or "-"
            what = f"hit {int(nd['hit_entity'])} t={float(nd['t']):.6g}" if nd["hit_entity"] >= 0 else "miss"
            if nd["hit_entity"] >= 0:
                what += f" {'exiting' if nd['exiting'] else 'entering'} ratio={float(nd['ratio']):.4g}"
            if int(nd["flags"]) & _capi.EUCL_TREE_SURFACE:
                what += f" surface=#{int(nd['surface_rgba8']):08x}"
            rgba = ", ".join(f"{float(c):.4f}" for c in nd["color"])
            lines.append(f"{'  ' * int(nd['level'])}[{j}] {TREE_KINDS[int(nd['kind'])]} level {int(nd['level'])} "
                         f"in {int(nd['medium'])}: {what} [{flags}] colour ({rgba})")
        if self.truncated:
            lines.append(f"... {self.count - len(self.nodes)} more nodes (capacity {len(self.nodes)})")
        return "\n".join(lines)


def default_tree_capacity(max_depth: int) -> int:
    """Nodes kept per tree unless asked otherwise: a full binary tree of max_depth + 1 levels, at most 4096."""
    return min(2 ** (int(max_depth) + 1) - 1, 4096)


def _tree_query(items: Sequence[int], capacity: int):
    """EuclTreeQuery over host arrays, and the arrays (kept alive by the caller): items, nodes, counts."""
    items = np.ascontiguousarray(items, dtype=np.uint32)
    capacity = int(capacity)
    if capacity < 1:
        raise ValueError("tree_capacity must be at least 1")
    if not 1 <= len(items) <= _capi.EUCL_TREE_MAX_ITEMS:
        raise ValueError(f"trees: 1 .. {_capi.EUCL_TREE_MAX_ITEMS} items")
    if len(items) * capacity > _capi.EUCL_TREE_MAX_NODES:
        raise ValueError(f"trees: {len(items)} items x capacity {capacity} exceed {_capi.EUCL_TREE_MAX_NODES} nodes")
    nodes = np.zeros((len(items), capacity), TREE_NODE_DTYPE)
    counts = np.zeros(len(items), np.uint32)
    query = EuclTreeQuery(items=items.ctypes.data, n_items=len(items), capacity=capacity, nodes=nodes.ctypes.data,
                          counts=counts.ctypes.data)
    return query, (items, nodes, counts)


def _cell(value, extent: int, what: str) -> int:
    v = int(value)
    if not 0 <= v < extent:
        raise ValueError(f"tree {what} {v} out of range 0 .. {extent - 1}")
    return v


def _frame_table(cameras: Sequence[EuclCamera], times) -> C.Array:
    """EuclFrame[K] from K cameras and a time per frame (or one time for all)."""
    cameras = list(cameras)
    if not cameras:
        raise ValueError("render_frames needs at least one camera")
    if any(not isinstance(c, EuclCamera) for c in cameras):
        raise TypeError("cameras must be EuclCamera poses (e.g. Environment.camera.copy())")
    if np.ndim(times) == 0:
        times = [float(times)] * len(cameras)
    else:
        times = [float(t) for t in times]
        if len(times) != len(cameras):
            raise ValueError(f"{len(cameras)} cameras but {len(times)} times")
    table = (EuclFrame * len(cameras))()
    for k, (cam, t) in enumerate(zip(cameras, times)):
        table[k].camera = cam
        table[k].time_seconds = t
    return table


def _decode_image(path: Path) -> Tuple[int, int, bytes]:
    """Decodes to RGBA8, row 0 = top -- the layout `image::DynamicImage::get_pixel` exposes
    (alpha = 255 for RGB / L images, grey replicated)."""
    from PIL import Image

    with Image.open(path) as im:
        rgba = im.convert("RGBA")
        return rgba.width, rgba.height, rgba.tobytes()


def stats_to_dict(st: EuclStats) -> dict:
    levels = int(st.levels)
    return {
        "pixels": int(st.pixels), "segments": int(st.segments), "nodes": int(st.nodes),
        "level_counts": [int(st.level_counts[i]) for i in range(levels)], "levels": levels,
        "retries": int(st.retries), "launches": int(st.launches), "ray_grouping": int(st.ray_grouping), "ms_total": float(st.ms_total),
        "ms_raygen": float(st.ms_raygen), "ms_intersect": float(st.ms_intersect), "ms_shade": float(st.ms_shade),
        "ms_resolve": float(st.ms_resolve), "graph_replays": int(st.graph_replays),
    }


class Environment:
    """A parsed universe (Universe3 / Universe4).  Mirrors `trait Environment` (src/universe/mod.rs:289-360)."""

    def __init__(self, parsed_handle: int, texture_paths: Sequence[str]):
        self._parsed = C.c_void_p(parsed_handle)
        self._scenes: Dict[Tuple[int, str], C.c_void_p] = {}
        self.texture_paths = list(texture_paths)
        flat = lib().eucl_parsed_flat(self._parsed)
        self.camera: EuclCamera = flat.contents.camera.copy()  # pose the JSON constructs; mutable by the caller
        self.pipeline = EUCL_PIPELINE_WAVEFRONT
        # the reference's scalar type F: "f64" (default build) or "f32" (cargo feature `low_precision`, src/main.rs:46-49)
        self.precision = "f64"

    # -- reference API ---------------------------------------------------------------------------
    def max_depth(self) -> int:
        return int(self.camera.max_depth)

    def render(self, dimensions: Tuple[int, int], time: float = 0.0, threads: int = 0,
               context: Optional[SimulationContext] = None, *, device: int = 0, want_hit_ids: bool = False,
               band_rows: int = 0, band_rank: int = 0, band_world: int = 1, out: Optional[np.ndarray] = None,
               profile: bool = False, aovs=None, trees: Optional[Sequence[Tuple[int, int]]] = None,
               tree_capacity: Optional[int] = None) -> RawImage2d:
        """Environment::render.  `time` is seconds since start (the reference passes a Duration);
        `threads` is accepted for signature parity and ignored (the GPU schedules the pixels).
        `aovs`: per-pixel auxiliary planes to return in `.aovs` (names from AOV_NAMES, or a mapping name -> array to
        render into); the frame, hit ids and stats are the same with or without them.
        `trees`: pixels (x, y), row 0 at the bottom, whose ray trees to return in `.trees` (RayTree, in request order),
        keeping up to `tree_capacity` nodes each (default: default_tree_capacity(max_depth)); not with `aovs`."""
        del threads
        context = context or SimulationContext()
        width, height = int(dimensions[0]) // context.resolution, int(dimensions[1]) // context.resolution
        items = self._tree_items(trees, aovs, lambda c: _cell(c[1], height, "y") * width + _cell(c[0], width, "x"))
        opts = EuclRenderOpts(width=width, height=height, time_seconds=float(time), band_rows=band_rows,
                              band_rank=band_rank, band_world=band_world, pipeline=self.pipeline, compact_rows=0,
                              want_hit_ids=int(want_hit_ids), profile=int(profile))
        if out is None:
            out = np.zeros((height, width, 3), dtype=np.uint8)
        assert out.dtype == np.uint8 and out.size == height * width * 3 and out.flags["C_CONTIGUOUS"]
        hit = np.full((height, width), -3, dtype=np.int32) if want_hit_ids else None
        planes = _aov_arrays(aovs, (height, width), self.dim) if aovs else None
        stats = EuclStats()
        result = None
        if planes:
            table = _frame_table([self.camera], float(time))
            check(lib().eucl_render_aovs(self._device_scene(device), table, 1, C.byref(opts), out.ctypes.data,
                                         hit.ctypes.data if hit is not None else None,
                                         C.byref(_aov_struct({n: a.ctypes.data for n, a in planes.items()})), C.byref(stats)))
        elif items is not None:
            query, result = _tree_query(items, self._tree_capacity(tree_capacity, self.camera.max_depth))
            check(lib().eucl_render_trees(self._device_scene(device), _frame_table([self.camera], float(time)), 1, C.byref(opts),
                                          out.ctypes.data, hit.ctypes.data if hit is not None else None, C.byref(query),
                                          C.byref(stats)))
        else:
            check(lib().eucl_render(self._device_scene(device), C.byref(self.camera), C.byref(opts), out.ctypes.data,
                                    hit.ctypes.data if hit is not None else None, C.byref(stats)))
        return RawImage2d(out, width, height, hit_ids=hit, stats=stats_to_dict(stats), aovs=planes,
                          trees=self._ray_trees(result))

    # -- device-resident variant (inputs and outputs stay in HBM) --------------------------------
    def render_device(self, d_out_rgb8: int, dimensions: Tuple[int, int], time: float = 0.0, *, device: int = 0,
                      d_out_hit_ids: int = 0, band_rows: int = 0, band_rank: int = 0, band_world: int = 1,
                      compact_rows: bool = False, profile: bool = False, d_aovs: Optional[Mapping[str, int]] = None) -> dict:
        """render into device buffers.  `d_aovs`: name -> device pointer of each wanted AOV plane (layout of the hit ids)."""
        width, height = int(dimensions[0]), int(dimensions[1])
        opts = EuclRenderOpts(width=width, height=height, time_seconds=float(time), band_rows=band_rows,
                              band_rank=band_rank, band_world=band_world, pipeline=self.pipeline,
                              compact_rows=int(compact_rows), want_hit_ids=int(bool(d_out_hit_ids)),
                              profile=int(profile))
        stats = EuclStats()
        if d_aovs:
            aov = _device_aovs(d_aovs)
            check(lib().eucl_render_aovs_device(self._device_scene(device), _frame_table([self.camera], float(time)), 1,
                                                C.byref(opts), C.c_void_p(d_out_rgb8),
                                                C.c_void_p(d_out_hit_ids) if d_out_hit_ids else None, C.byref(aov), C.byref(stats)))
        else:
            check(lib().eucl_render_device(self._device_scene(device), C.byref(self.camera), C.byref(opts),
                                           C.c_void_p(d_out_rgb8), C.c_void_p(d_out_hit_ids) if d_out_hit_ids else None,
                                           C.byref(stats)))
        return stats_to_dict(stats)

    # -- many frames per call: camera paths and animations -------------------------------------------
    def render_frames(self, dimensions: Tuple[int, int], cameras: Sequence[EuclCamera], times=0.0,
                      context: Optional[SimulationContext] = None, *, device: int = 0, want_hit_ids: bool = False,
                      out: Optional[np.ndarray] = None, profile: bool = False, aovs=None,
                      trees: Optional[Sequence[Tuple[int, int, int]]] = None, tree_capacity: Optional[int] = None) -> RawFrames:
        """Renders one frame per camera pose in ONE call (eucl_render_frames): frame k equals
        `render(dimensions, times[k])` with `self.camera` set to `cameras[k]`, bit for bit.  `times` is one time for
        every frame or a sequence of one per frame.  Batching pays the fixed cost of a frame once per call.
        `aovs` as for `render`; plane k of the result belongs to frame k.  `trees`: pixels (k, x, y) of frame k, as for
        `render`."""
        table = _frame_table(cameras, times)
        context = context or SimulationContext()
        width, height = int(dimensions[0]) // context.resolution, int(dimensions[1]) // context.resolution
        k = len(table)
        items = self._tree_items(trees, aovs, lambda c: ((_cell(c[0], k, "frame") * height + _cell(c[2], height, "y")) * width
                                                         + _cell(c[1], width, "x")))
        if out is None:
            out = np.zeros((k, height, width, 3), dtype=np.uint8)
        if out.dtype != np.uint8 or out.shape != (k, height, width, 3) or not out.flags["C_CONTIGUOUS"]:
            raise ValueError(f"out must be a C-contiguous uint8 array of shape {(k, height, width, 3)}")
        opts = EuclRenderOpts(width=width, height=height, pipeline=self.pipeline, want_hit_ids=int(want_hit_ids),
                              profile=int(profile))
        hit = np.full((k, height, width), -3, dtype=np.int32) if want_hit_ids else None
        planes = _aov_arrays(aovs, (k, height, width), self.dim) if aovs else None
        stats = EuclStats()
        result = None
        if planes:
            check(lib().eucl_render_aovs(self._device_scene(device), table, k, C.byref(opts), out.ctypes.data,
                                         hit.ctypes.data if hit is not None else None,
                                         C.byref(_aov_struct({n: a.ctypes.data for n, a in planes.items()})), C.byref(stats)))
        elif items is not None:
            query, result = _tree_query(items, self._tree_capacity(tree_capacity, table[0].camera.max_depth))
            check(lib().eucl_render_trees(self._device_scene(device), table, k, C.byref(opts), out.ctypes.data,
                                          hit.ctypes.data if hit is not None else None, C.byref(query), C.byref(stats)))
        else:
            check(lib().eucl_render_frames(self._device_scene(device), table, k, C.byref(opts), out.ctypes.data,
                                           hit.ctypes.data if hit is not None else None, C.byref(stats)))
        return RawFrames(out, width, height, hit_ids=hit, stats=stats_to_dict(stats), aovs=planes, trees=self._ray_trees(result))

    def render_frames_device(self, d_out_rgb8: int, dimensions: Tuple[int, int], cameras: Sequence[EuclCamera],
                             times=0.0, *, device: int = 0, d_out_hit_ids: int = 0, profile: bool = False,
                             d_aovs: Optional[Mapping[str, int]] = None) -> dict:
        """render_frames into device buffers: K * height * width * 3 bytes (and K * height * width int32 hit ids, and the
        AOV planes of `d_aovs`, name -> device pointer)."""
        table = _frame_table(cameras, times)
        width, height = int(dimensions[0]), int(dimensions[1])
        opts = EuclRenderOpts(width=width, height=height, pipeline=self.pipeline, want_hit_ids=int(bool(d_out_hit_ids)),
                              profile=int(profile))
        stats = EuclStats()
        if d_aovs:
            aov = _device_aovs(d_aovs)
            check(lib().eucl_render_aovs_device(self._device_scene(device), table, len(table), C.byref(opts),
                                                C.c_void_p(d_out_rgb8), C.c_void_p(d_out_hit_ids) if d_out_hit_ids else None,
                                                C.byref(aov), C.byref(stats)))
        else:
            check(lib().eucl_render_frames_device(self._device_scene(device), table, len(table), C.byref(opts),
                                                  C.c_void_p(d_out_rgb8), C.c_void_p(d_out_hit_ids) if d_out_hit_ids else None,
                                                  C.byref(stats)))
        return stats_to_dict(stats)

    # -- caller-supplied rays: custom projections, picking, probes -----------------------------------
    def trace_rays(self, origins, directions, time: float = 0.0, *, max_depth: Optional[int] = None,
                   width: Optional[int] = None, device: int = 0, want_hit_ids: bool = True, aovs=None,
                   out: Optional[np.ndarray] = None, profile: bool = False, trees=None,
                   tree_capacity: Optional[int] = None) -> RawRays:
        """Traces one ray per origin / direction pair (eucl_trace_rays): arrays of shape (..., dim), converted to
        float64.  Directions are used as given (not normalised).  Ray i gives what a pixel whose camera ray is
        (origins[i], directions[i]) gives -- its RGB8 value, primary hit and AOV planes -- and an origin in no entity gives
        the checkerboard of grid cell (i % width, i // width).  `width` (rays per grid row) defaults to the last leading
        dimension of an (H, W, dim) grid and to 1 for a flat (N, dim) list; `max_depth` to the camera's.  Tracing the
        camera's own rays of a w x h frame with width w reproduces `render((w, h), time)` bit for bit.
        `trees`: rays whose ray trees to return in `.trees` (RayTree, in request order), each a flat ray index or an index
        tuple into the rays' leading shape; `tree_capacity` as for `render`; not with `aovs`."""
        o, d, lead = _ray_arrays(origins, directions, self.dim)
        n = int(np.prod(lead, dtype=np.int64))
        items = self._tree_items(trees, aovs, lambda c: (int(np.ravel_multi_index(tuple(int(v) for v in c), lead))
                                                         if isinstance(c, (tuple, list)) else _cell(c, n, "ray index")))
        if width is None:
            width = lead[-1] if len(lead) >= 2 else 1
        rays = _ray_struct(n, width, self.camera.max_depth if max_depth is None else max_depth, self.pipeline, time, profile,
                           o.ctypes.data, d.ctypes.data)
        if out is None:
            out = np.zeros(lead + (3,), dtype=np.uint8)
        if out.dtype != np.uint8 or out.shape != lead + (3,) or not out.flags["C_CONTIGUOUS"]:
            raise ValueError(f"out must be a C-contiguous uint8 array of shape {lead + (3,)}")
        hit = np.full(lead, -3, dtype=np.int32) if want_hit_ids else None
        planes = _aov_arrays(aovs, lead, self.dim) if aovs else None
        stats = EuclStats()
        result = None
        if items is not None:
            query, result = _tree_query(items, self._tree_capacity(tree_capacity, rays.max_depth))
            check(lib().eucl_trace_ray_trees(self._device_scene(device), C.byref(rays), out.ctypes.data,
                                             hit.ctypes.data if hit is not None else None, C.byref(query), C.byref(stats)))
        else:
            aov = C.byref(_aov_struct({k: a.ctypes.data for k, a in planes.items()})) if planes else None
            check(lib().eucl_trace_rays(self._device_scene(device), C.byref(rays), out.ctypes.data,
                                        hit.ctypes.data if hit is not None else None, aov, C.byref(stats)))
        return RawRays(out, hit_ids=hit, stats=stats_to_dict(stats), aovs=planes, trees=self._ray_trees(result))

    def trace_rays_device(self, d_origins: int, d_directions: int, n: int, d_out_rgb8: int, time: float = 0.0, *,
                          max_depth: Optional[int] = None, width: int = 1, device: int = 0, d_out_hit_ids: int = 0,
                          d_aovs: Optional[Mapping[str, int]] = None, profile: bool = False) -> dict:
        """trace_rays with DEVICE arrays: `n` rays of `dim` float64 each at d_origins / d_directions, n * 3 bytes of RGB8,
        n int32 hit ids and the AOV planes of `d_aovs` (name -> device pointer).  Returns the stats."""
        rays = _ray_struct(int(n), width, self.camera.max_depth if max_depth is None else max_depth, self.pipeline, time,
                           profile, int(d_origins), int(d_directions))
        stats = EuclStats()
        aov = C.byref(_device_aovs(d_aovs)) if d_aovs else None
        check(lib().eucl_trace_rays_device(self._device_scene(device), C.byref(rays), C.c_void_p(d_out_rgb8),
                                           C.c_void_p(d_out_hit_ids) if d_out_hit_ids else None, aov, C.byref(stats)))
        return stats_to_dict(stats)

    def trace_path_unknown(self, location: Sequence[float], direction: Sequence[float], distance: float, *,
                           device: int = 0) -> Optional[Tuple[list, list]]:
        """Universe::trace_path_unknown (src/universe/mod.rs:273-286): the point reached by travelling
        `distance` along `direction` through the universe (voids stretch or shrink the step) and the
        direction of travel there; None when `location` lies in no entity.  The reference's cameras
        move with this call (d3/entity/camera.rs:223-243)."""
        dim = self.dim
        loc = (C.c_double * dim)(*[float(v) for v in location[:dim]])
        dirv = (C.c_double * dim)(*[float(v) for v in direction[:dim]])
        out_l, out_d = (C.c_double * dim)(), (C.c_double * dim)()
        status = lib().eucl_trace_path(self._device_scene(device), loc, dirv, float(distance), out_l, out_d)
        if status == 1:
            return None
        check(status)
        return list(out_l), list(out_d)

    def move_camera(self, direction: Sequence[float], distance: float, *, device: int = 0) -> bool:
        """Translates `self.camera.location` like the translation part of the reference's camera
        `update` (d3/entity/camera.rs:223-243): normalised direction, trace_path_unknown, new location.
        (The reference additionally turns the view when the void bends the path; it labels that code
        "not tested", and it is not reproduced here.)  Returns False when the camera is in no entity."""
        dim = self.dim
        step = camera_step(direction, distance, dim)
        if step is None:
            return True
        res = self.trace_path_unknown([self.camera.location[k] for k in range(dim)], step[0], step[1], device=device)
        if res is None:
            return False
        for k in range(dim):
            self.camera.location[k] = res[0][k]
        return True

    # -- universe queries in bulk: one device call for many points or walkers -------------------------
    def locate(self, points, *, device: int = 0) -> np.ndarray:
        """Universe::material_at (mod.rs:229-251) of every point (eucl_locate_points): an array of shape (..., dim) gives
        int32 (...), the first entity in list order whose shape contains the point, -1 when none does."""
        p, lead = _point_array(points, self.dim, "points")
        out = np.empty(lead, np.int32)
        check(lib().eucl_locate_points(self._device_scene(device), p.ctypes.data, out.size, out.ctypes.data))
        return out

    def locate_device(self, d_points: int, n: int, d_out: int, *, device: int = 0) -> None:
        """locate with DEVICE arrays: n points of `dim` float64 at d_points, n int32 entities at d_out."""
        check(lib().eucl_locate_points_device(self._device_scene(device), C.c_void_p(int(d_points)), int(n),
                                              C.c_void_p(int(d_out))))

    def trace_paths(self, locations, directions, distances, steps: int = 1, *,
                    device: int = 0) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
        """Universe::trace_path_unknown for many walkers, `steps` steps each (eucl_trace_paths): locations and directions
        of shape (..., dim), distances a scalar or of the leading shape.  Step j starts where step j-1 ended and walks the
        walker's own distance along its own direction (used as given), as `move_camera` steps a camera.  Returns
        (locations (..., steps, dim), directions (..., steps, dim), status (..., steps)): status 1 moved; 0 the step's
        start lies in no entity (the walker stays, direction NaN, later steps alike); -1 more than 100000 surface
        crossings (NaN, and the walker stops)."""
        loc, lead = _point_array(locations, self.dim, "locations")
        dirs, dlead = _point_array(directions, self.dim, "directions")
        if dlead != lead:
            raise ValueError(f"locations {loc.shape} and directions {dirs.shape} must have the same shape")
        dist = np.asarray(distances, dtype=np.float64)
        if dist.shape not in ((), lead):
            raise ValueError(f"distances must be a scalar or of shape {lead}, got {dist.shape}")
        dist = np.ascontiguousarray(np.broadcast_to(dist, lead))
        steps = int(steps)
        n = int(np.prod(lead, dtype=np.int64))
        if steps < 1 or n * steps > 0x7FFFFFFF:
            raise ValueError("trace_paths needs steps >= 1 and n * steps <= 2^31 - 1")
        out_loc = np.empty(lead + (steps, self.dim), np.float64)
        out_dir = np.empty_like(out_loc)
        status = np.empty(lead + (steps,), np.int32)
        check(lib().eucl_trace_paths(self._device_scene(device), loc.ctypes.data, dirs.ctypes.data, dist.ctypes.data, n, steps,
                                     out_loc.ctypes.data, out_dir.ctypes.data, status.ctypes.data))
        return out_loc, out_dir, status

    def trace_paths_device(self, d_locations: int, d_directions: int, d_distances: int, n: int, steps: int,
                           d_out_locations: int, d_out_status: int, d_out_directions: int = 0, *, device: int = 0) -> None:
        """trace_paths with DEVICE arrays: n walkers (dim float64 locations and directions, one float64 distance each),
        outputs [n][steps] ([n][steps][dim] float64 locations and, unless 0, directions; int32 status)."""
        check(lib().eucl_trace_paths_device(self._device_scene(device), C.c_void_p(int(d_locations)),
                                            C.c_void_p(int(d_directions)), C.c_void_p(int(d_distances)), int(n), int(steps),
                                            C.c_void_p(int(d_out_locations)),
                                            C.c_void_p(int(d_out_directions)) if d_out_directions else None,
                                            C.c_void_p(int(d_out_status))))

    # The view-turning part of the reference's camera `update` (d3/entity/camera.rs:94-145,303-350;
    # d4/entity/camera.rs:68-130).  The reference derives the angles from mouse deltas and held keys;
    # here the caller passes them (radians).  `kind` names the reference camera type being mimicked.
    def rotate_yaw(self, angle: float, kind: str = "PitchYawCamera3") -> None:
        check(lib().eucl_camera_rotate_yaw(C.byref(self.camera), float(angle), 0 if kind == "PitchYawCamera3" else 1))

    def rotate_pitch(self, angle: float, kind: str = "PitchYawCamera3") -> None:
        check(lib().eucl_camera_rotate_pitch(C.byref(self.camera), float(angle), 1 if kind == "PitchYawCamera3" else 0))

    def rotate_roll(self, angle: float) -> None:
        check(lib().eucl_camera_rotate_roll(C.byref(self.camera), float(angle)))

    def rotate_plane4(self, axis_a: int, axis_b: int, angle: float) -> None:
        """FreeCamera4: rotation in the plane of two camera axes (0 forward, 1 left, 2 up, 3 ana)."""
        check(lib().eucl_camera_rotate_plane4(C.byref(self.camera), int(axis_a), int(axis_b), float(angle)))

    # -- plumbing ----------------------------------------------------------------------------------
    @staticmethod
    def _tree_items(trees, aovs, item_of) -> Optional[List[int]]:
        """The virtual-frame cells of the requested trees (None: no tree call); ValueError with AOVs or for an empty or
        out-of-range request."""
        if trees is None:
            return None
        if aovs:
            raise ValueError("trees and aovs cannot be asked for in one call")
        items = [item_of(c) for c in trees]
        if not items:
            raise ValueError("trees names no item")
        return items

    @staticmethod
    def _tree_capacity(tree_capacity: Optional[int], max_depth: int) -> int:
        return default_tree_capacity(max_depth) if tree_capacity is None else int(tree_capacity)

    def _ray_trees(self, result) -> Optional[List[RayTree]]:
        if result is None:
            return None
        _, nodes, counts = result
        cap = nodes.shape[1]
        return [RayTree(nodes[i, :min(int(c), cap)], int(c), self.dim, self.precision) for i, c in enumerate(counts)]

    @property
    def flat(self) -> EuclFlatScene:
        return lib().eucl_parsed_flat(self._parsed).contents

    @property
    def dim(self) -> int:
        return int(self.flat.dim)

    def _device_scene(self, device: int) -> C.c_void_p:
        key = (device, self.precision)
        if key not in self._scenes:
            if self.precision not in ("f64", "f32"):
                raise ValueError("precision must be 'f64' or 'f32'")
            handle = C.c_void_p()
            check(lib().eucl_scene_create_precision(lib().eucl_parsed_flat(self._parsed), device,
                                                    _capi.EUCL_PRECISION_F32 if self.precision == "f32" else _capi.EUCL_PRECISION_F64,
                                                    C.byref(handle)))
            self._scenes[key] = handle
        return self._scenes[key]

    def set_texture(self, slot: int, width: int, height: int, rgba8: bytes) -> None:
        """Fills texture slot `slot` with decoded RGBA8 pixels (row 0 = top); for callers that decode
        images themselves.  Must happen before the first render."""
        assert len(rgba8) == width * height * 4
        check(lib().eucl_parsed_set_texture(self._parsed, slot, width, height, rgba8))

    def memory(self, device: int = 0) -> dict:
        """Device memory this environment's scene holds for frames: node arena, index lists, node capacity."""
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        check(lib().eucl_scene_memory(self._device_scene(device), C.byref(a), C.byref(b), C.byref(c)))
        return {"arena_bytes": a.value, "list_bytes": b.value, "node_capacity": c.value}

    def set_stream(self, cuda_stream: int, device: int = 0) -> None:
        """Runs this environment's kernels on `cuda_stream` (e.g. torch.cuda.current_stream().cuda_stream)."""
        check(lib().eucl_scene_set_stream(self._device_scene(device), C.c_void_p(cuda_stream)))

    def close(self) -> None:
        for handle in self._scenes.values():
            lib().eucl_scene_destroy(handle)
        self._scenes.clear()
        if self._parsed:
            lib().eucl_parsed_destroy(self._parsed)
            self._parsed = C.c_void_p()

    def __del__(self):  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass


@dataclass
class Parser:
    """scene::Parser (src/scene.rs:554-1478).  `resource_root` plays the role of the reference's
    working directory for the `./resources/...` texture paths (src/scene.rs:1050-1072)."""
    resource_root: Union[str, os.PathLike, None] = None
    texture_substitutes: Dict[str, str] = field(default_factory=lambda: dict(DEFAULT_TEXTURE_SUBSTITUTES))

    @classmethod
    def default(cls, resource_root: Union[str, os.PathLike, None] = None) -> "Parser":
        return cls(resource_root=resource_root)

    def _resolve(self, texture_path: str) -> Path:
        root = Path(self.resource_root) if self.resource_root is not None else Path.cwd()
        p = root / texture_path
        if not p.exists() and p.name in self.texture_substitutes:
            p = p.with_name(self.texture_substitutes[p.name])
        if not p.exists():
            raise FileNotFoundError(f"texture `{texture_path}` not found under {root}")
        return p

    def parse(self, json_text: str, *, load_textures: bool = True) -> Environment:
        handle = C.c_void_p()
        check(lib().eucl_scene_parse(json_text.encode("utf-8"), C.byref(handle)))
        n = lib().eucl_parsed_texture_count(handle)
        paths = [lib().eucl_parsed_texture_path(handle, k).decode("utf-8") for k in range(n)]
        if load_textures:
            try:
                for slot, tex in enumerate(paths):
                    w, h, data = _decode_image(self._resolve(tex))
                    check(lib().eucl_parsed_set_texture(handle, slot, w, h, data))
            except Exception:
                lib().eucl_parsed_destroy(handle)
                raise
        return Environment(handle.value, paths)

    def parse_file(self, path: Union[str, os.PathLike], **kw) -> Environment:
        return self.parse(Path(path).read_text(), **kw)
