"""Universe queries in bulk (eucl_locate_points*, eucl_trace_paths*; Environment.locate, Environment.trace_paths): many
points located and many walkers moved through the universe in one device call.  On the GPU, bit for bit: locate equals the
CPU oracle's Universe::material_at (oracle/oracle_features.cc) and what a render decides about a ray's origin, trace_paths
equals eucl_trace_path called once per walker and step and the oracle's trace_path_unknown, the host variants equal the
device variants across chunk boundaries, a query leaves a render's graph replay alone, and the tool's camera path and
entity sections equal their definitions.  The CPU tests cover the ABI, the argument checks and the tool's options."""
import ctypes as C
import math
import sys
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb
import oracle_api
from test_negated_rooms import SHAPES as NEGATED_ROOMS, load as load_negated, scene as negated_scene

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import eucl_render  # noqa: E402

REFERENCE = sorted(p.stem for p in (ROOT / "assets" / "scenes").glob("*.json"))
EUCL_ERR_INVALID_ARGUMENT = -1
CHUNK = 1 << 18  # kQueryChunk of api_device.cu: items a host query stages per round trip


def load(name, precision="f64"):
    if name in ("no_void_3d", "csg_mix_3d"):
        env = eb.Parser.default(resource_root=ROOT).parse_file(ROOT / "tests" / "scenes" / f"{name}.json")
    elif name in NEGATED_ROOMS:
        env = load_negated(negated_scene(NEGATED_ROOMS[name]))
    else:
        env = eb.load_reference_scene(name)
    env.precision = precision
    return env


def variant(precision):
    return "f32" if precision == "f32" else "det"


def same(a, b) -> bool:
    """Equal bit patterns, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.kind != "f":
        return np.array_equal(a, b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint64), b[~nb].view(np.uint64))


def scene_extent(env) -> float:
    """A radius that holds the camera and every bounded sphere of the scene."""
    flat, dim = env.flat, env.dim
    ext = max(10.0, float(np.linalg.norm([env.camera.location[k] for k in range(dim)])))
    for i in range(flat.n_prims):
        p = flat.prims[i]
        if p.kind == 1 and math.isfinite(p.s0):
            ext = max(ext, float(np.linalg.norm([p.v0[k] for k in range(dim)])) + abs(p.s0))
    return ext


def query_points(env, n, seed):
    """Random points in and around the scene, points on its spheres and planes (boundary ties), and points with NaN and
    infinite components."""
    rng = np.random.default_rng(seed)
    dim, ext, flat = env.dim, scene_extent(env), env.flat
    pts = [rng.uniform(-1.3 * ext, 1.3 * ext, (n, dim)),
           np.array([env.camera.location[k] for k in range(dim)]) + rng.normal(0.0, 0.1 * ext, (n, dim))]
    for i in range(flat.n_prims):
        p = flat.prims[i]
        v0 = np.array([p.v0[k] for k in range(dim)])
        if p.kind == eb._capi.PRIM_SPHERE and math.isfinite(p.s0):
            axes = np.concatenate([np.eye(dim), -np.eye(dim)])
            pts.append(v0 + p.s0 * axes)  # exactly on the surface along the axes
            u = rng.normal(size=(8, dim))
            pts.append(v0 + p.s0 * u / np.linalg.norm(u, axis=1, keepdims=True))
        elif p.kind in (eb._capi.PRIM_HALFSPACE, eb._capi.PRIM_HYPERPLANE) and v0.any():
            q = rng.uniform(-ext, ext, (8, dim))
            for c in (p.s0, -p.s0):  # on the plane n . x = c, whichever sign the table stores
                pts.append(q - ((q @ v0 - c) / (v0 @ v0))[:, None] * v0)
    special = rng.uniform(-ext, ext, (6 * dim, dim))
    for j, v in enumerate([np.nan, np.inf, -np.inf] * 2 * dim):
        special[j, (j // 3) % dim] = v
    pts.append(special)
    pts.append(np.full((1, dim), np.nan))
    return np.ascontiguousarray(np.concatenate(pts))


# ---------------------------------------------------------------------------------------------------------- GPU: locate

@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name", REFERENCE + ["csg_mix_3d", "no_void_3d"] + sorted(NEGATED_ROOMS))
def test_locate_equals_oracle(built_lib, name, precision):
    env = load(name, precision)
    pts = query_points(env, 3000, seed=len(name))
    got = env.locate(pts)
    want = oracle_api.locate(env, pts, variant(precision))
    assert got.dtype == np.int32 and got.shape == (len(pts),)
    bad = np.flatnonzero(got != want)
    assert not len(bad), f"{len(bad)} points differ, first {pts[bad[0]]}: {got[bad[0]]} vs {want[bad[0]]}"
    if precision == "f64":  # the f64 oracle's own material_at hook
        lib = oracle_api.lib("det")
        for i in range(0, len(pts), 97):
            assert got[i] == lib.oracle_material_at(C.byref(env.flat), oracle_api.darr(pts[i]))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["no_void_3d", "3d_room", "4d_room", "box_room"])
def test_locate_equals_the_renderers_origin_decision(built_lib, name):
    """A ray's hit id is -2 exactly where its origin is in no entity, and a tree's root medium is the origin's entity."""
    env = load(name)
    rng = np.random.default_rng(3)
    dim, ext = env.dim, scene_extent(env)
    w, h = 24, 16
    for shift in (0.0, 0.5 * ext, 2.0 * ext):  # the camera's rays from places in and out of the entities
        cam = env.camera.copy()
        cam.location[0] += shift
        o, d = oracle_api.camera_rays(env, w, h, camera=cam)
        o = o + rng.normal(0.0, 0.2 * ext, (h, w, 1)) * (np.arange(dim) == 1)  # a different origin per ray
        res = env.trace_rays(o, d, max_depth=2)
        located = env.locate(o)
        assert np.array_equal(res.hit_ids == -2, located == -1)
    o = rng.uniform(-1.3 * ext, 1.3 * ext, (300, dim))
    d = rng.normal(size=(300, dim))
    items = list(range(0, 300, 7))
    res = env.trace_rays(o, d, max_depth=1, trees=items)
    located = env.locate(o[items])
    assert [int(t.nodes["medium"][0]) for t in res.trees] == located.tolist()


# ----------------------------------------------------------------------------------------------------- GPU: trace_paths

def walkers(env, n, seed):
    rng = np.random.default_rng(seed)
    dim, ext = env.dim, scene_extent(env)
    loc = rng.uniform(-0.8 * ext, 0.8 * ext, (n, dim))
    loc[:, 2] = rng.uniform(-3.5, 5.0, n)
    loc[: n // 4] = rng.uniform(-3.0 * ext, 3.0 * ext, (n // 4, dim))  # some far out: in no entity where the scene ends
    d = rng.normal(size=(n, dim))
    d *= rng.uniform(0.3, 3.0, (n, 1)) / np.linalg.norm(d, axis=1, keepdims=True)  # used as given, not normalised
    dist = rng.uniform(0.1, 40.0, n)
    return loc, d, dist


def chained(env, loc, d, dist, steps, oracle_variant=None):
    """`steps` trace_path_unknown calls with the move_camera rule (each from where the last ended, the walker's own
    direction and distance), by the single-walker entry point or by the oracle."""
    out_l, out_d, status = np.full((steps, env.dim), np.nan), np.full((steps, env.dim), np.nan), np.zeros(steps, np.int32)
    here = list(loc)
    for j in range(steps):
        if oracle_variant:
            res = oracle_api.trace_path(env, here, d, float(dist), variant=oracle_variant)
        else:
            res = env.trace_path_unknown(here, d, float(dist))
        if res is None:
            out_l[j:], status[j:] = here, 0
            break
        here = res[0]
        out_l[j], out_d[j], status[j] = res[0], res[1], 1
    return out_l, out_d, status


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name", ["3d_hallways", "3d_fresnel", "3d_room", "4d_room", "4d_cylinders", "no_void_3d"])
def test_trace_paths_one_step_equals_single_calls(built_lib, name, precision):
    env = load(name, precision)
    loc, d, dist = walkers(env, 150, seed=11)
    got_l, got_d, got_s = env.trace_paths(loc, d, dist)
    assert got_l.shape == (150, 1, env.dim) and got_d.shape == got_l.shape and got_s.shape == (150, 1)
    for i in range(150):
        single = env.trace_path_unknown(loc[i], d[i], dist[i])
        oracle = oracle_api.trace_path(env, loc[i], d[i], dist[i], variant=variant(precision))
        assert (single is None) == (oracle is None)
        if single is None:
            assert got_s[i, 0] == 0 and same(got_l[i, 0], loc[i]) and np.isnan(got_d[i, 0]).all()
        else:
            assert got_s[i, 0] == 1
            assert same(got_l[i, 0], single[0]) and same(got_d[i, 0], single[1])
            assert same(got_l[i, 0], oracle[0]) and same(got_d[i, 0], oracle[1])
    if name == "no_void_3d":
        assert (got_s == 0).any() and (got_s == 1).any()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name", ["3d_hallways", "4d_room", "no_void_3d"])
def test_trace_paths_steps_equal_chained_calls(built_lib, name, precision):
    env = load(name, precision)
    steps = 6
    loc, d, dist = walkers(env, 40, seed=5)
    dist *= 0.3
    got_l, got_d, got_s = env.trace_paths(loc, d, dist, steps=steps)
    for i in range(40):
        want = chained(env, loc[i], d[i], dist[i], steps)
        assert same(got_l[i], want[0]) and same(got_d[i], want[1]) and np.array_equal(got_s[i], want[2]), f"walker {i}"
        if i % 5 == 0:
            ref = chained(env, loc[i], d[i], dist[i], steps, oracle_variant=variant(precision))
            assert same(got_l[i], ref[0]) and same(got_d[i], ref[1]) and np.array_equal(got_s[i], ref[2])


# --------------------------------------------------------------------------------------------- GPU: shapes and chunking

class DeviceArrays:
    def __init__(self, **arrays):
        import torch

        self.t = {k: torch.from_numpy(np.ascontiguousarray(v)).cuda() for k, v in arrays.items()}

    def ptr(self, k):
        return self.t[k].data_ptr()

    def get(self, k):
        import torch

        torch.cuda.synchronize()
        return self.t[k].cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 513, CHUNK + 77])
def test_locate_sizes_and_device_variant(built_lib, n):
    env = load("3d_room")
    pts = query_points(env, max(n // 2, 1), seed=n)[:n]
    if len(pts) < n:
        pts = np.resize(pts, (n, env.dim))
    got = env.locate(pts)
    dev = DeviceArrays(points=pts, out=np.full(n, -7, np.int32))
    env.locate_device(dev.ptr("points"), n, dev.ptr("out"))
    assert np.array_equal(dev.get("out"), got)
    sample = np.arange(0, n, max(1, n // 3000))
    assert np.array_equal(got[sample], oracle_api.locate(env, pts[sample]))
    assert env.locate(pts[0]).shape == () and env.locate(pts[0]) == got[0]
    grid = query_points(env, 12, seed=1)[:12].reshape(3, 4, env.dim)
    assert np.array_equal(env.locate(grid), env.locate(grid.reshape(12, env.dim)).reshape(3, 4))


@pytest.mark.gpu
@pytest.mark.parametrize("n,steps", [(1, 1), (1, 5), (1000, 1), (CHUNK + 77, 1), (CHUNK // 3 * 2 + 5, 3)])
def test_trace_paths_sizes_and_device_variant(built_lib, n, steps):
    env = load("3d_hallways")
    loc, d, dist = walkers(env, n, seed=n + steps)
    got_l, got_d, got_s = env.trace_paths(loc, d, dist, steps=steps)
    nan = np.full((n, steps, env.dim), np.nan)
    dev = DeviceArrays(loc=loc, d=d, dist=dist, out_l=nan, out_d=nan, status=np.full((n, steps), 7, np.int32))
    env.trace_paths_device(dev.ptr("loc"), dev.ptr("d"), dev.ptr("dist"), n, steps, dev.ptr("out_l"), dev.ptr("status"),
                           dev.ptr("out_d"))
    assert same(dev.get("out_l"), got_l) and same(dev.get("out_d"), got_d) and np.array_equal(dev.get("status"), got_s)
    for i in np.linspace(0, n - 1, min(n, 12)).astype(int):  # walkers of every chunk against the single-walker calls
        want = chained(env, loc[i], d[i], dist[i], steps)
        assert same(got_l[i], want[0]) and same(got_d[i], want[1]) and np.array_equal(got_s[i], want[2])
    # without directions, and with one distance for every walker
    dev2 = DeviceArrays(out_l=nan, status=np.zeros((n, steps), np.int32))
    env.trace_paths_device(dev.ptr("loc"), dev.ptr("d"), dev.ptr("dist"), n, steps, dev2.ptr("out_l"), dev2.ptr("status"))
    assert same(dev2.get("out_l"), got_l) and np.array_equal(dev2.get("status"), got_s)
    m = min(n, 50)
    one_l, _, one_s = env.trace_paths(loc[:m], d[:m], 2.5, steps=steps)
    want_l, _, want_s = env.trace_paths(loc[:m], d[:m], np.full(m, 2.5), steps=steps)
    assert same(one_l, want_l) and np.array_equal(one_s, want_s)


# ----------------------------------------------------------------------------------------------- GPU: no side effects

@pytest.mark.gpu
def test_queries_leave_the_render_graph_alone(built_lib):
    env = load("3d_room")
    w, h = 64, 40
    for _ in range(12):  # the scene settles its ray-grouping mode, then the render runs as a graph
        ref = env.render((w, h), 0.5, want_hit_ids=True)
        if ref.stats["graph_replays"]:
            break
    assert ref.stats["graph_replays"] > 0
    loc, d, dist = walkers(env, 5000, seed=2)
    env.locate(loc)
    env.trace_paths(loc, d, dist, steps=2)
    after = env.render((w, h), 0.5, want_hit_ids=True)
    assert after.stats["graph_replays"] > 0
    assert np.array_equal(after.data, ref.data) and np.array_equal(after.hit_ids, ref.hit_ids)


# ------------------------------------------------------------------------------------------- GPU: invalid arguments

@pytest.mark.gpu
def test_invalid_arguments(built_lib):
    env = load("4d_room")
    s = env._device_scene(0)
    p = np.zeros((4, 4))
    out = np.zeros(4, np.int32)
    o = np.zeros((4, 3, 4))
    st = np.zeros((4, 3), np.int32)
    dist = np.zeros(4)
    a = lambda x: x.ctypes.data
    lib = built_lib
    for fn in (lib.eucl_locate_points, lib.eucl_locate_points_device):
        assert fn(s, None, 4, a(out)) == EUCL_ERR_INVALID_ARGUMENT
        assert fn(s, a(p), 4, None) == EUCL_ERR_INVALID_ARGUMENT
        assert fn(s, a(p), 0, a(out)) == EUCL_ERR_INVALID_ARGUMENT
        assert fn(None, a(p), 4, a(out)) == EUCL_ERR_INVALID_ARGUMENT
    for fn in (lib.eucl_trace_paths, lib.eucl_trace_paths_device):
        args = [a(p), a(p), a(dist), 4, 3, a(o), a(o), a(st)]
        for k in (0, 1, 2, 5, 7):  # every required pointer
            bad = list(args)
            bad[k] = None
            assert fn(s, *bad) == EUCL_ERR_INVALID_ARGUMENT, k
        for n, steps in ((0, 3), (4, 0), (1 << 16, 1 << 15), (0x7FFFFFFF, 2)):
            bad = list(args)
            bad[3], bad[4] = n, steps
            assert fn(s, *bad) == EUCL_ERR_INVALID_ARGUMENT, (n, steps)
    # the scene still works, and the largest legal call shape is accepted by the checks
    assert env.locate(p).shape == (4,)
    with pytest.raises(ValueError):
        env.locate(np.zeros((4, 3)))
    with pytest.raises(ValueError):
        env.trace_paths(p, p, dist, steps=0)


# ---------------------------------------------------------------------------------------------------------- GPU: tool

@pytest.mark.gpu
def test_tool_camera_path_is_one_call_and_equals_move_camera(built_lib, tmp_path, monkeypatch):
    scene = ROOT / "assets" / "scenes" / "3d_hallways.json"
    size = (48, 32)
    calls = []
    real = eb.Environment.trace_paths

    def counted(self, *a, **kw):
        calls.append(kw.get("steps"))
        return real(self, *a, **kw)

    monkeypatch.setattr(eb.Environment, "trace_paths", counted)
    monkeypatch.setattr(eb.Environment, "trace_path_unknown", lambda *a, **kw: pytest.fail("a per-frame path call"))
    eucl_render.main([str(scene), str(tmp_path / "f_%04d.ppm"), "--size", *map(str, size), "--frames", "8",
                      "--move", "0", "0.5", "0", "--yaw", "0.05"])
    assert calls == [7]
    monkeypatch.undo()
    env = load("3d_hallways")
    cameras = []
    for k in range(8):
        if k:
            assert env.move_camera([0.0, 0.5, 0.0], 1.0)
            env.rotate_yaw(0.05)
        cameras.append(env.camera.copy())
    assert len({tuple(c.location) for c in cameras}) == 8
    frames = env.render_frames(size, cameras)
    for k in range(8):
        frames.frame(k).save(tmp_path / f"loop_{k}.ppm")
        assert (tmp_path / f"f_{k:04d}.ppm").read_bytes() == (tmp_path / f"loop_{k}.ppm").read_bytes(), f"frame {k}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room"])
def test_tool_section_equals_locate(built_lib, tmp_path, name):
    scene = ROOT / "assets" / "scenes" / f"{name}.json"
    w, h, extent = 40, 30, 24.0
    eucl_render.main([str(scene), str(tmp_path / "s.png"), "--size", str(w), str(h), "--section", str(extent)])
    entity = np.load(tmp_path / "s.entity.npy")
    env = load(name)
    cam, dim = env.camera, env.dim
    f = np.array(cam.forward[:dim])
    if dim == 3:  # the camera's right axis, as its rays use it
        right = np.cross(f, np.array(cam.up[:dim]))
        right = right / np.linalg.norm(right)
    else:
        right = -np.array(cam.left[:dim])
    xs = (np.arange(w) + 0.5 - w / 2) * (extent / w)
    ys = (np.arange(h) + 0.5 - h / 2) * (extent / w)
    pts = np.array(cam.location[:dim]) + xs[None, :, None] * right + ys[:, None, None] * f
    assert entity.dtype == np.int32 and entity.shape == (h, w)
    assert np.array_equal(entity, oracle_api.locate(env, pts))
    assert len(np.unique(entity)) > 1
    from PIL import Image

    img = np.asarray(Image.open(tmp_path / "s.png"))
    assert np.array_equal(img, eucl_render.section_image(entity)[::-1])


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_query_symbols_and_prototypes(built_lib):
    from euclider_b200 import _capi

    for name, nargs in (("eucl_locate_points", 4), ("eucl_locate_points_device", 4), ("eucl_trace_paths", 9),
                        ("eucl_trace_paths_device", 9)):
        assert hasattr(built_lib, name)
        restype, argtypes = _capi.PROTOTYPES[name]
        assert restype is C.c_int and len(argtypes) == nargs
        assert getattr(built_lib, name).argtypes == argtypes
    # checked before any device is touched: a null scene is an invalid argument, GPU or not
    pts, out = np.zeros((2, 3)), np.zeros(2, np.int32)
    assert built_lib.eucl_locate_points(None, pts.ctypes.data, 2, out.ctypes.data) == EUCL_ERR_INVALID_ARGUMENT
    assert built_lib.eucl_trace_paths(None, pts.ctypes.data, pts.ctypes.data, pts.ctypes.data, 2, 1, pts.ctypes.data, None,
                                      out.ctypes.data) == EUCL_ERR_INVALID_ARGUMENT


def test_python_argument_checks(built_lib):
    env = eb.load_reference_scene("3d_room")  # every check fails before a device scene is made
    for bad in (np.zeros((5, 4)), np.zeros((0, 3)), np.zeros(()), [["a", "b", "c"]]):
        with pytest.raises(ValueError):
            env.locate(bad)
    p = np.zeros((5, 3))
    for kw in (dict(locations=np.zeros((5, 4)), directions=p, distances=1.0),
               dict(locations=p, directions=np.zeros((4, 3)), distances=1.0),
               dict(locations=p, directions=p, distances=np.ones(4)),
               dict(locations=np.zeros((0, 3)), directions=np.zeros((0, 3)), distances=1.0),
               dict(locations=p, directions=p, distances=1.0, steps=0),
               dict(locations=p, directions=p, distances=1.0, steps=1 << 29)):
        with pytest.raises(ValueError):
            env.trace_paths(**kw)


def test_camera_step_is_move_cameras_normalisation():
    unit, dist = eb.camera_step([0.0, 3.0, 4.0], 2.0, 3)
    assert unit == [0.0, 0.6, 0.8] and dist == 10.0
    assert eb.camera_step([0, 0, 0], 1.0, 3) is None
    assert eb.camera_step([1, 2, 2, 7], 1.0, 3) == ([1 / 3, 2 / 3, 2 / 3], 3.0)


def test_tool_section_option_parsing():
    a = eucl_render.parse_args(["s.json", "o.png", "--section", "12.5"])
    assert a.section == 12.5
    for bad in (["--aov", "depth"], ["--inspect", "1,1"], ["--frames", "2"], ["--move", "0", "1", "0"],
                ["--projection", "equirect"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o_%04d.png" if "--frames" in bad else "o.png", "--section", "10", *bad])
    for bad in (["--section", "0"], ["--section", "-1"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o.png", *bad])


def test_section_plane_geometry():
    cam = eb.EuclCamera()
    cam.dim = 3
    for k, v in enumerate((1.0, 2.0, 3.0)):
        cam.location[k] = v
    cam.forward[0], cam.up[2] = 1.0, 1.0  # right = forward x up = -y
    pts = eucl_render.section_points(cam, 3, 4, 2, 8.0)
    assert pts.shape == (2, 4, 3)
    assert np.array_equal(pts[0, 0], [1.0 - 1.0, 2.0 + 3.0, 3.0])  # bottom-left centre: x -1 (forward), y +3 (left)
    assert np.array_equal(pts[1, 3], [1.0 + 1.0, 2.0 - 3.0, 3.0])
    img = eucl_render.section_image(np.array([[-1, 0, 17]], np.int32))
    assert img.dtype == np.uint8 and (img[0, 0] == 0).all() and (img[0, 1] == eucl_render.SECTION_PALETTE[0]).all()
    assert (img[0, 2] == eucl_render.SECTION_PALETTE[17 % len(eucl_render.SECTION_PALETTE)]).all()
