"""Caller-supplied rays (eucl_trace_rays*, Environment.trace_rays): the camera's own rays reproduce eucl_render bit for
bit, and arbitrary rays -- unnormalised, degenerate, starting in no entity or inside a LinearSpace void -- equal the CPU
oracle's definition (oracle/oracle_features.cc) bit for bit, any NaN equal to any NaN, through every part of the machinery a
frame uses (chunks, retries, split pipelines, graph replays).  The CPU tests cover the ABI struct, the oracle exports, the
Python argument checks, the equirect geometry and the tool's --projection option."""
import ctypes as C
import math
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb
import oracle_api

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import eucl_render  # noqa: E402

ALL = eb.AOV_NAMES
SCENES = sorted(p.stem for p in (ROOT / "assets" / "scenes").glob("*.json"))
COUNTED = ("pixels", "segments", "nodes", "level_counts")
EUCL_OK, EUCL_ERR_INVALID_ARGUMENT, EUCL_ERR_SCENE_LIMIT = 0, -1, -21


def load(name):
    if name in ("no_void_3d", "csg_mix_3d"):
        return eb.Parser.default(resource_root=ROOT).parse_file(ROOT / "tests" / "scenes" / f"{name}.json")
    return eb.load_reference_scene(name)


def pipeline_id(name):
    return eb.EUCL_PIPELINE_MEGAKERNEL if name == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT


def same(a, b) -> bool:
    """Equal bit patterns, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    if a.dtype.kind != "f":
        return np.array_equal(a, b)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def assert_same_result(got, rgb, hit, planes, what=""):
    assert np.array_equal(got.data, rgb), f"{what}RGB differs"
    assert np.array_equal(got.hit_ids, hit), f"{what}hit ids differ"
    for n in ALL:
        assert same(got.aovs[n], planes[n]), f"{what}{n} differs"


def scene_extent(env) -> float:
    """A radius that holds the camera and every bounded sphere of the scene."""
    flat, dim = env.flat, env.dim
    ext = max(10.0, float(np.linalg.norm([env.camera.location[k] for k in range(dim)])))
    for i in range(flat.n_prims):
        p = flat.prims[i]
        if p.kind == 1 and math.isfinite(p.s0):
            ext = max(ext, float(np.linalg.norm([p.v0[k] for k in range(dim)])) + abs(p.s0))
    return ext


def random_rays(env, n, seed):
    """Half the origins near the camera, half spread over and beyond the scene; random unnormalised directions with
    lengths from 1e-3 to 1e3."""
    rng = np.random.default_rng(seed)
    dim, ext = env.dim, scene_extent(env)
    loc = np.array([env.camera.location[k] for k in range(dim)])
    near = loc + rng.normal(0.0, 0.05 * ext, (n // 2, dim))
    far = rng.uniform(-1.5 * ext, 1.5 * ext, (n - n // 2, dim))
    origins = np.concatenate([near, far])
    d = rng.normal(size=(n, dim))
    d *= (10.0 ** rng.uniform(-3, 3, (n, 1))) / np.linalg.norm(d, axis=1, keepdims=True)
    return origins, d


def check_rays_oracle(env, origins, directions, time=0.0, max_depth=None, width=None, variant="det"):
    """One trace_rays call with every plane against the oracle; returns it."""
    got = env.trace_rays(origins, directions, time, max_depth=max_depth, width=width, aovs=ALL)
    rgb, hit, planes, st = oracle_api.trace_rays(env, origins, directions, time=time, max_depth=max_depth, width=width,
                                                 variant=variant)
    assert_same_result(got, rgb, hit, planes)
    assert got.stats["segments"] == st["segments"] and got.stats["nodes"] == st["nodes"]
    assert got.stats["level_counts"] == st["level_counts"]
    assert got.stats["pixels"] == int(np.prod(np.shape(origins)[:-1]))
    return got


def check_identity(env, size, time=0.5, variant="det", camera=None):
    """The camera's w x h rays (oracle ray_vector) traced with width w == the render, bit for bit, counted stats too."""
    w, h = size
    saved = env.camera.copy()
    if camera is not None:
        env.camera = camera.copy()
    try:
        img = env.render(size, time, want_hit_ids=True, aovs=ALL)
        o, d = oracle_api.camera_rays(env, w, h, variant=variant)
        got = env.trace_rays(o, d, time, aovs=ALL)
    finally:
        env.camera = saved
    assert got.data.shape == (h, w, 3)
    assert_same_result(got, img.data, img.hit_ids, img.aovs)
    assert {k: got.stats[k] for k in COUNTED} == {k: img.stats[k] for k in COUNTED}
    return got


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", SCENES)
def test_camera_rays_equal_render(built_lib, name, pipeline):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    check_identity(env, (96, 54))


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_fresnel", "4d_cylinders"])
def test_camera_rays_equal_render_f32(built_lib, name, pipeline):
    env = load(name)
    env.precision = "f32"
    env.pipeline = pipeline_id(pipeline)
    check_identity(env, (96, 54), variant="f32")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_hallways"])
def test_camera_rays_of_moved_and_turned_cameras(built_lib, name):
    env = load(name)
    step = [0.0] * env.dim
    step[0], step[1] = 0.05, 0.15
    env.move_camera(step, 2.0)
    if env.dim == 3:
        env.rotate_yaw(0.3)
        env.rotate_pitch(-0.1)
    else:
        env.rotate_plane4(0, 1, 0.2)
        env.rotate_plane4(2, 3, 0.1)
    check_identity(env, (61, 37), time=0.75)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_camera_in_no_entity_gives_the_checkerboard(built_lib, pipeline):
    env = load("no_void_3d")
    env.pipeline = pipeline_id(pipeline)
    got = check_identity(env, (37, 23))
    assert (got.hit_ids == -2).all() and got.stats["nodes"] == 0 and got.stats["pixels"] == 37 * 23


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCENES + ["csg_mix_3d"])
def test_random_rays_equal_oracle(built_lib, name):
    env = load(name)
    o, d = random_rays(env, 3000, seed=sum(name.encode()))
    check_rays_oracle(env, o, d, time=1.25)


@pytest.mark.gpu
@pytest.mark.parametrize("depth", [0, 1, 10, 16])
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "csg_mix_3d"])
def test_random_rays_all_builds(built_lib, name, precision, pipeline, depth):
    env = load(name)
    env.precision = precision
    env.pipeline = pipeline_id(pipeline)
    o, d = random_rays(env, 2000, seed=depth + 7)
    check_rays_oracle(env, o, d, time=0.5, max_depth=depth, variant="det" if precision == "f64" else "f32")


def degenerate_rays(env):
    dim = env.dim
    loc = [env.camera.location[k] for k in range(dim)]
    unit = [1.0] + [0.0] * (dim - 1)
    rays = [(loc, [0.0] * dim), (loc, [math.nan] + [0.5] * (dim - 1)), (loc, [math.inf] + [0.0] * (dim - 1)),
            (loc, [-math.inf, 1.0] + [0.0] * (dim - 2)), ([math.nan] * dim, unit), ([math.inf] + loc[1:], unit),
            (loc, [1e-300] * dim), (loc, [1e300] * dim)]
    flat = env.flat
    for i in range(flat.n_prims):  # origins exactly on sphere surfaces, looking along and across the normal
        p = flat.prims[i]
        if p.kind == 1 and math.isfinite(p.s0):
            c = [p.v0[k] for k in range(dim)]
            on = [c[0] + p.s0] + c[1:]
            rays += [(on, unit), (on, [-1.0] + [0.0] * (dim - 1)), (on, [0.0, 1.0] + [0.0] * (dim - 2))]
    return rays


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "csg_mix_3d"])
def test_degenerate_rays(built_lib, name, pipeline):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    rays = degenerate_rays(env)
    if name == "csg_mix_3d":  # the LinearSpace void's boundary (the cuboid around (6, 0, 0)) and points across it
        for x in (5.0, 5.5, 6.5, 7.0):
            for dx in (1.0, -1.0, 0.0):
                rays.append(([x, 0.0, 0.0], [dx, 0.25, 0.0]))
    o = np.array([r[0] for r in rays], np.float64)
    d = np.array([r[1] for r in rays], np.float64)
    check_rays_oracle(env, o, d)


@pytest.mark.gpu
def test_flat_list_equals_grid(built_lib):
    env = load("no_void_3d")  # traced and untraced rays
    o, d = random_rays(env, 48 * 40, seed=3)
    o[: len(o) // 2] = [10.0, 0.0, 0.5]  # half of the origins inside the sphere
    grid = env.trace_rays(o.reshape(40, 48, 3), d.reshape(40, 48, 3), aovs=ALL)
    flat = env.trace_rays(o, d, aovs=ALL)
    traced = flat.hit_ids != -2
    assert traced.any() and (~traced).any()
    assert np.array_equal(grid.hit_ids.ravel(), flat.hit_ids)
    assert np.array_equal(grid.data.reshape(-1, 3)[traced], flat.data[traced])
    for n in ALL:
        assert same(grid.aovs[n].reshape(flat.aovs[n].shape), flat.aovs[n]), n
    assert {k: grid.stats[k] for k in COUNTED} == {k: flat.stats[k] for k in COUNTED}
    check_rays_oracle(env, o.reshape(40, 48, 3), d.reshape(40, 48, 3))
    check_rays_oracle(env, o, d, width=16)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room"])
def test_split_pipelines_equal_one(built_lib, monkeypatch, name):
    env = load(name)
    o, d = random_rays(env, 256 * 288, seed=11)
    o, d = o.reshape(288, 256, -1), d.reshape(288, 256, -1)
    results = []
    for split in (1, 2, 3):
        monkeypatch.setenv("EUCL_SPLIT", str(split))
        results.append(env.trace_rays(o, d, 0.5, aovs=ALL))
    for r in results[1:]:
        assert_same_result(r, results[0].data, results[0].hit_ids, results[0].aovs)
        assert {k: r.stats[k] for k in COUNTED} == {k: results[0].stats[k] for k in COUNTED}
    rows = slice(100, 104)  # a sample against the oracle
    rgb, hit, planes, _ = oracle_api.trace_rays(env, o[rows], d[rows], time=0.5)
    assert np.array_equal(results[2].data[rows], rgb) and np.array_equal(results[2].hit_ids[rows], hit)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_pixels", [200, 777])
def test_chunk_boundaries_inside_the_list(built_lib, monkeypatch, chunk_pixels):
    env = load("3d_room")
    o, d = random_rays(env, 2400, seed=5)
    ref = env.trace_rays(o, d, aovs=ALL)
    monkeypatch.setenv("EUCL_CHUNK_PIXELS", str(chunk_pixels))
    for width in (1, 48):
        got = check_rays_oracle(env, o.reshape(-1, width, 3) if width > 1 else o, d.reshape(-1, width, 3) if width > 1 else d)
        traced = ref.hit_ids != -2  # (checkerboard cells depend on the width)
        assert np.array_equal(got.data.reshape(-1, 3)[traced], ref.data[traced])
        assert np.array_equal(got.hit_ids.ravel(), ref.hit_ids)


@pytest.mark.gpu
def test_forced_arena_retry(built_lib, monkeypatch):
    env = load("3d_fresnel_2")
    o, d = oracle_api.camera_rays(env, 48, 31)
    plain = env.trace_rays(o, d, aovs=ALL)
    monkeypatch.setenv("EUCL_ARENA_FACTOR_X10", "11")
    tight = load("3d_fresnel_2")
    got = tight.trace_rays(o, d, aovs=ALL, profile=True)
    assert got.stats["retries"] > 0
    assert_same_result(got, plain.data, plain.hit_ids, plain.aovs)
    check_rays_oracle(tight, o, d)


class DeviceRays:
    """Device copies of rays and device outputs (torch tensors)."""

    def __init__(self, n, dim):
        import torch

        self.o = torch.zeros((n, dim), dtype=torch.float64, device="cuda")
        self.d = torch.zeros_like(self.o)
        self.rgb = torch.zeros((n, 3), dtype=torch.uint8, device="cuda")
        self.hit = torch.zeros(n, dtype=torch.int32, device="cuda")
        self.planes = {"depth": torch.zeros(n, dtype=torch.float32, device="cuda"),
                       "position": torch.zeros((n, dim), dtype=torch.float32, device="cuda"),
                       "normal": torch.zeros((n, dim), dtype=torch.float32, device="cuda"),
                       "segments": torch.zeros(n, dtype=torch.int32, device="cuda"),
                       "levels": torch.zeros(n, dtype=torch.int32, device="cuda")}

    def trace(self, env, o, d, **kw):
        import torch

        self.o.copy_(torch.from_numpy(o))
        self.d.copy_(torch.from_numpy(d))
        for t in [self.rgb, self.hit, *self.planes.values()]:
            t.fill_(-7)
        return env.trace_rays_device(self.o.data_ptr(), self.d.data_ptr(), len(o), self.rgb.data_ptr(),
                                     d_out_hit_ids=self.hit.data_ptr(), d_aovs={n: t.data_ptr() for n, t in self.planes.items()},
                                     **kw)

    def result(self):
        planes = {n: t.cpu().numpy() for n, t in self.planes.items()}
        planes["segments"], planes["levels"] = planes["segments"].view(np.uint32), planes["levels"].view(np.uint32)
        return eb.RawRays(self.rgb.cpu().numpy(), hit_ids=self.hit.cpu().numpy(), aovs=planes)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_device_entry_and_graph_replay(built_lib, pipeline):
    env = load("4d_room")
    env.pipeline = pipeline_id(pipeline)
    n = 3000
    dev = DeviceRays(n, env.dim)
    replays = []
    for seed in (1, 2, 3):  # the same buffers, new contents: a replayed graph must read them
        o, d = random_rays(env, n, seed)
        st = dev.trace(env, o, d, time=0.5)
        replays.append(st["graph_replays"])
        rgb, hit, planes, ost = oracle_api.trace_rays(env, o, d, time=0.5)
        assert_same_result(dev.result(), rgb, hit, planes, what=f"seed {seed}: ")
        assert st["level_counts"] == ost["level_counts"]
    assert replays[2] > 0


@pytest.mark.gpu
def test_host_entry_graph_replay(built_lib):
    env = load("3d_room")
    replays = []
    for seed in (4, 5, 6):
        o, d = random_rays(env, 2500, seed)
        got = check_rays_oracle(env, o, d, time=0.25)
        replays.append(got.stats["graph_replays"])
    assert replays[2] > 0


@pytest.mark.gpu
def test_render_and_trace_rays_alternate(built_lib):
    env = load("3d_room")
    w, h = 64, 40
    o, d = oracle_api.camera_rays(env, w, h)
    o2, d2 = o.copy(), d[::-1].copy()  # the same grid, other rays
    # the scene settles its ray-grouping mode (no graphs while it measures), then the render runs as a graph
    for _ in range(12):
        ref = env.render((w, h), 0.5, want_hit_ids=True)
        if ref.stats["graph_replays"]:
            break
    assert ref.stats["graph_replays"] > 0
    ref2 = env.trace_rays(o2, d2, 0.5)
    assert not np.array_equal(ref.data, ref2.data)
    # Both kinds of call write the scene's staging frame with equal time, depth and grid size, and the scene keeps one
    # graph: a ray call made while the render's graph is held, or a render made while a ray call's graph is held, that
    # replayed the other's graph would return the other's picture.  Each kind does replay its own graph in this sequence.
    replays = {"render": 0, "rays": 0}
    for step, kind in enumerate(["rays", "render", "rays", "render", "rays", "rays", "render", "render", "rays"]):
        if kind == "render":
            got, want = env.render((w, h), 0.5, want_hit_ids=True), ref
        else:
            got, want = env.trace_rays(o2, d2, 0.5), ref2
        assert np.array_equal(got.data, want.data) and np.array_equal(got.hit_ids, want.hit_ids), f"step {step} ({kind})"
        replays[kind] += got.stats["graph_replays"]
    assert replays["render"] > 0 and replays["rays"] > 0, replays
    # and the camera's own rays, which equal the render, in the same alternation
    assert np.array_equal(env.trace_rays(o, d, 0.5).data, ref.data)


@pytest.mark.gpu
def test_with_and_without_planes(built_lib):
    env = load("4d_room")
    o, d = random_rays(env, 1000, seed=21)
    full = env.trace_rays(o, d, aovs=ALL)
    plain = env.trace_rays(o, d)
    assert plain.aovs is None
    assert np.array_equal(full.data, plain.data) and np.array_equal(full.hit_ids, plain.hit_ids)
    assert {k: full.stats[k] for k in COUNTED} == {k: plain.stats[k] for k in COUNTED}
    some = env.trace_rays(o, d, aovs=["depth", "levels"], want_hit_ids=False)
    assert some.hit_ids is None and set(some.aovs) == {"depth", "levels"}
    assert same(some.aovs["depth"], full.aovs["depth"]) and same(some.aovs["levels"], full.aovs["levels"])
    # an EuclAovs without any plane counts as none
    out = np.zeros((len(o), 3), np.uint8)
    rays = eb.EuclRays(origins=o.ctypes.data, directions=d.ctypes.data, n=len(o), width=1, max_depth=10)
    assert eb.lib().eucl_trace_rays(env._device_scene(0), C.byref(rays), out.ctypes.data, None, C.byref(eb.EuclAovs()),
                                    C.byref(eb.EuclStats())) == EUCL_OK
    assert np.array_equal(out, full.data)


@pytest.mark.gpu
def test_invalid_arguments_are_rejected(built_lib):
    env = load("3d_room")
    scene = env._device_scene(0)
    lib = eb.lib()
    o = np.zeros((12, 3))
    d = np.ones((12, 3))
    out = np.full((12, 3), 77, np.uint8)

    def call(rgb=out, **kw):
        fields = dict(origins=o.ctypes.data, directions=d.ctypes.data, n=12, width=1, max_depth=10, pipeline=0)
        fields.update(kw)
        r = eb.EuclRays(**fields)
        return lib.eucl_trace_rays(scene, C.byref(r), rgb.ctypes.data if rgb is not None else None, None, None,
                                   C.byref(eb.EuclStats()))

    for kw in [dict(n=0), dict(n=0x80000000), dict(origins=None), dict(directions=None), dict(rgb=None), dict(width=5),
               dict(width=24), dict(max_depth=64), dict(max_depth=0xFFFFFFFF), dict(pipeline=2)]:
        assert call(**kw) == EUCL_ERR_INVALID_ARGUMENT, kw
    assert (out == 77).all()  # rejected before any device work
    assert lib.eucl_trace_rays(scene, None, out.ctypes.data, None, None, None) == EUCL_ERR_INVALID_ARGUMENT
    r = eb.EuclRays(origins=o.ctypes.data, directions=d.ctypes.data, n=12, width=1, max_depth=10)
    assert lib.eucl_trace_rays_device(scene, C.byref(r), None, None, None, None) == EUCL_ERR_INVALID_ARGUMENT
    assert call(pipeline=1, max_depth=25) == EUCL_ERR_SCENE_LIMIT
    assert call(width=4) == EUCL_OK and call(width=0) == EUCL_OK and (out != 77).any()


@pytest.mark.gpu
def test_tool_equirect(built_lib, tmp_path):
    from PIL import Image

    scene = ROOT / "assets" / "scenes" / "3d_room.json"
    w, h = 64, 32
    subprocess.run([sys.executable, str(ROOT / "tools" / "eucl_render.py"), str(scene), str(tmp_path / "pano.png"), "--size",
                    str(w), str(h), "--projection", "equirect", "--time", "0.5"], check=True, capture_output=True)
    img = np.asarray(Image.open(tmp_path / "pano.png").convert("RGB"))[::-1]
    env = load("3d_room")
    ref = env.trace_rays(*eb.equirect_rays(env.camera, w, h), 0.5)
    assert np.array_equal(img, ref.data)


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_rays_struct_layout():
    from euclider_b200._capi import EuclRays

    assert C.sizeof(EuclRays) == 48
    names = ["origins", "directions", "n", "width", "max_depth", "pipeline", "time_seconds", "profile", "_pad"]
    assert [getattr(EuclRays, n).offset for n in names] == [0, 8, 16, 20, 24, 28, 32, 40, 44]


def test_new_kernels_are_in_the_library(built_lib):
    import shutil

    import test_kernel_resources as kr

    if not Path(kr.CUOBJDUMP).exists() and not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump (CUDA toolkit) not installed")
    from euclider_b200 import _capi

    names = list(kr.resource_usage(_capi.LIB_PATH))
    for tag in ("k_raygen_rays", "k_megakernel_rays", "k_megakernel_rays_aov"):
        for ns in ("_ZN4euclANON", "_ZN8eucl_fANON"):  # the f64 and the f32 build, D = 3 and 4 each
            assert sum(1 for k in names if k.startswith(ns + tag + "I")) == 2, (ns, tag)


def test_python_argument_checks():
    env = eb.load_reference_scene("3d_room")
    o = np.zeros((6, 3))
    with pytest.raises(ValueError):
        env.trace_rays(o, np.zeros((5, 3)))  # shape mismatch
    with pytest.raises(ValueError):
        env.trace_rays(np.zeros((6, 4)), np.zeros((6, 4)))  # 4-D rays, 3-D scene
    with pytest.raises(ValueError):
        env.trace_rays(np.zeros((0, 3)), np.zeros((0, 3)))  # no rays
    with pytest.raises(ValueError):
        env.trace_rays(o, o, width=4)  # 4 does not divide 6
    with pytest.raises(ValueError):
        env.trace_rays(o, o, aovs=["depth", "albedo"])
    with pytest.raises(ValueError):
        env.trace_rays(o, o, aovs={"depth": np.zeros(5, np.float32)})
    with pytest.raises(ValueError):
        env.trace_rays(o, o, out=np.zeros((6, 4), np.uint8))
    with pytest.raises(ValueError):
        env.trace_rays(o, o, max_depth=64)
    with pytest.raises(ValueError):
        env.trace_rays_device(0, 0, 10, 0, width=3)
    with pytest.raises(ValueError):
        env.trace_rays_device(0, 0, 10, 0, d_aovs={"depht": 1})


@pytest.mark.parametrize("name", ["3d_room", "4d_room"])
def test_equirect_geometry(name):
    env = eb.load_reference_scene(name)
    cam, dim = env.camera, env.dim
    f = np.array(cam.forward[:dim])
    u = np.array(cam.up[:dim])
    w, h = 9, 5
    o, d = eb.equirect_rays(cam, w, h)
    assert o.shape == d.shape == (h, w, dim) and o.dtype == d.dtype == np.float64
    assert np.allclose(o, np.array(cam.location[:dim]))
    assert np.allclose(np.linalg.norm(d, axis=-1), 1.0)  # orthonormal camera axes: unit directions
    assert np.allclose(d[h // 2, w // 2], f)  # the centre of an odd grid looks forward
    assert np.dot(d[-1, w // 2], u) > 0 > np.dot(d[0, w // 2], u)  # row 0 at the bottom
    # the seam: the first and last columns sit half a column from phi = -pi and +pi, mirror images of each other
    if dim == 3:
        left = -np.cross(f, u) / np.linalg.norm(np.cross(f, u))
    else:
        left = np.array(cam.left[:dim])
    mid = d[h // 2]
    phi = np.arctan2(-mid @ left, mid @ f)
    assert np.allclose(phi, 2 * np.pi * ((np.arange(w) + 0.5) / w - 0.5))
    assert np.isclose(phi[0], -np.pi + np.pi / w) and np.isclose(phi[-1], np.pi - np.pi / w)
    assert np.allclose(mid[0] @ f, mid[-1] @ f) and np.allclose(mid[0] @ left, -(mid[-1] @ left))


def test_tool_projection_option_parsing():
    assert eucl_render.parse_args(["s.json", "o.png"]).projection == "perspective"
    assert eucl_render.parse_args(["s.json", "o.png", "--projection", "equirect"]).projection == "equirect"
    for bad in (["--projection", "fisheye"], ["--projection", "equirect", "--frames", "2", "o_%d.png"],
                ["--projection", "equirect", "--yaw", "0.1"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o.png", *bad])


@pytest.mark.parametrize("variant", ["det", "f32"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room"])
def test_oracle_camera_rays_equal_ray_vector(oracle, name, variant):
    env = load(name)
    w, h = 13, 7
    o, d = oracle_api.camera_rays(env, w, h, variant=variant)
    assert np.array_equal(o, np.broadcast_to(o[0, 0], o.shape))
    if variant == "f32":  # float rays, widened
        assert np.array_equal(d.astype(np.float32).astype(np.float64), d)
        return
    lib = oracle.lib("det")
    for y in range(h):
        for x in range(w):
            v = (C.c_double * env.dim)()
            lib.oracle_ray_vector(C.byref(env.flat), C.byref(env.camera), x, y, w, h, v)
            assert list(v) == list(d[y, x]), (x, y)


@pytest.mark.parametrize("name,size,variant", [("3d_room", (40, 23), "det"), ("4d_room", (32, 18), "det"),
                                               ("3d_room", (32, 18), "f32"), ("no_void_3d", (24, 16), "det"),
                                               ("csg_mix_3d", (32, 18), "det")])
def test_oracle_trace_rays_of_camera_rays_equals_render(name, size, variant):
    env = load(name)
    w, h = size
    o, d = oracle_api.camera_rays(env, w, h, variant=variant)
    rgb, hit, planes, st = oracle_api.trace_rays(env, o, d, time=0.5, variant=variant)
    rgb0, hit0, planes0, st0 = oracle_api.render_aovs(env, w, h, time=0.5, variant=variant)
    assert np.array_equal(rgb, rgb0) and np.array_equal(hit, hit0)
    for n in ALL:
        assert same(planes[n], planes0[n]), n
    assert st == st0
