"""Per-pixel auxiliary outputs (eucl_render_aovs*, Environment.render(..., aovs=...)): depth, position and normal of the
primary hit and the segments and levels of each pixel's ray tree equal the CPU oracle's planes (oracle/oracle_features.cc)
bit for bit -- any NaN equals any NaN -- in every layout a render has (batches, bands, compact rows, two pipelines,
chunks, retries, graph replays), on both pipelines and precisions; and asking for them changes nothing else.  The CPU
tests cover the ABI struct, the oracle's own consistency, the Python argument checks and the tool's --aov option."""
import ctypes as C
import os
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
EUCL_ERR_INVALID_ARGUMENT = -1
SENTINEL = {"depth": -7.0, "position": -7.0, "normal": -7.0, "segments": 0xDEADBEEF, "levels": 0xDEADBEEF}


def load(name):
    if name == "no_void_3d":
        return eb.Parser.default(resource_root=ROOT).parse_file(ROOT / "tests" / "scenes" / "no_void_3d.json")
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


def assert_planes(got: dict, want: dict, names=ALL, what=""):
    for n in names:
        assert same(got[n], want[n]), f"{what}{n} differs"


def sentinel_planes(lead, dim, names=ALL):
    out = {}
    for n in names:
        per_dim = n in ("position", "normal")
        dtype = np.uint32 if n in ("segments", "levels") else np.float32
        out[n] = np.full(lead + ((dim,) if per_dim else ()), SENTINEL[n], dtype=dtype)
    return out


def camera_path(env, k):
    cams = []
    step = [0.0] * env.dim
    step[0], step[1] = 0.05, 0.15
    for i in range(k):
        if i:
            env.move_camera(step, 1.0)
            if env.dim == 3:
                env.rotate_yaw(0.07)
                env.rotate_pitch(-0.03)
            else:
                env.rotate_plane4(0, 1, 0.06)
                env.rotate_plane4(2, 3, 0.04)
        cams.append(env.camera.copy())
    return cams


def check_oracle(env, size, time=0.0, camera=None, variant="det", rows=None):
    """One AOV render against the oracle (and its plain twin): returns the render."""
    w, h = size
    saved = env.camera.copy()
    if camera is not None:
        env.camera = camera.copy()
    try:
        img = env.render(size, time, want_hit_ids=True, aovs=ALL)
        plain = env.render(size, time, want_hit_ids=True)
    finally:
        env.camera = saved
    rgb, hit, planes, st = oracle_api.render_aovs(env, w, h, time=time, camera=camera, variant=variant, rows=rows)
    r0, r1 = rows or (0, h)
    assert np.array_equal(img.data[r0:r1], rgb) and np.array_equal(img.hit_ids[r0:r1], hit), "frame differs from the oracle"
    assert_planes({n: a[r0:r1] for n, a in img.aovs.items()}, planes)
    # asking for AOVs changes nothing else
    assert np.array_equal(img.data, plain.data) and np.array_equal(img.hit_ids, plain.hit_ids)
    assert {k: img.stats[k] for k in COUNTED} == {k: plain.stats[k] for k in COUNTED}
    assert int(img.aovs["segments"].sum(dtype=np.uint64)) == img.stats["segments"]
    assert int(img.aovs["levels"].max()) <= int((camera or env.camera).max_depth) + 1
    return img


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", SCENES)
def test_reference_scenes_equal_oracle(built_lib, name):
    check_oracle(load(name), (96, 54), time=0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_fresnel_2", "4d_cylinders"])
def test_megakernel_equals_wavefront(built_lib, name):
    env = load(name)
    wave = env.render((61, 37), 0.25, want_hit_ids=True, aovs=ALL)
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL
    mega = check_oracle(env, (61, 37), time=0.25)
    assert np.array_equal(mega.data, wave.data)
    assert_planes(mega.aovs, wave.aovs)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_fresnel"])
def test_low_precision_equals_f32_oracle(built_lib, name, pipeline):
    env = load(name)
    env.precision = "f32"
    env.pipeline = pipeline_id(pipeline)
    check_oracle(env, (53, 31), time=1.5, variant="f32")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_hallways"])
def test_moved_and_turned_cameras(built_lib, name):
    env = load(name)
    for cam in camera_path(env, 4)[1:]:
        check_oracle(env, (45, 27), time=0.75, camera=cam)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_camera_in_no_entity(built_lib, pipeline):
    env = load("no_void_3d")
    env.pipeline = pipeline_id(pipeline)
    img = check_oracle(env, (37, 23))
    assert (img.hit_ids == -2).all()
    assert np.isnan(img.aovs["depth"]).all() and np.isnan(img.aovs["position"]).all() and np.isnan(img.aovs["normal"]).all()
    assert (img.aovs["segments"] == 0).all() and (img.aovs["levels"] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("depth", [0, 1, 16])
def test_max_depth(built_lib, pipeline, depth):
    env = load("3d_room")
    env.pipeline = pipeline_id(pipeline)
    env.camera.max_depth = depth
    img = check_oracle(env, (48, 27), time=0.5)
    if depth == 0:
        assert (img.aovs["depth"] == np.inf).all() and np.isnan(img.aovs["normal"]).all()
        assert (img.aovs["levels"] == 1).all() and (img.aovs["segments"] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["no_void_3d", "3d_room", "4d_room"])
def test_batch_frames_equal_single_renders(built_lib, pipeline, name):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    if name == "no_void_3d":  # untraced (camera in no entity) and traced frames in one batch
        cams = []
        for loc in [(0, 0, 0), (10, 0, 0), (10.5, 0.5, 0), (0, 0, 0)]:
            cam = env.camera.copy()
            for k in range(3):
                cam.location[k] = loc[k]
            cams.append(cam)
    else:
        cams = camera_path(env, 4)
    times = [0.0, 0.5, 1.0, 1.5]
    batch = env.render_frames((37, 23), cams, times, want_hit_ids=True, aovs=ALL)
    plain = env.render_frames((37, 23), cams, times, want_hit_ids=True)
    assert np.array_equal(batch.data, plain.data) and np.array_equal(batch.hit_ids, plain.hit_ids)
    assert {k: batch.stats[k] for k in COUNTED} == {k: plain.stats[k] for k in COUNTED}
    saved = env.camera.copy()
    for k, (cam, t) in enumerate(zip(cams, times)):
        env.camera = cam.copy()
        one = env.render((37, 23), t, aovs=ALL)
        assert_planes(batch.frame(k).aovs, one.aovs, what=f"frame {k}: ")
    env.camera = saved
    assert int(batch.aovs["segments"].sum(dtype=np.uint64)) == batch.stats["segments"]


@pytest.mark.gpu
@pytest.mark.parametrize("world,band", [(3, 8), (2, 16)])
def test_band_split_host_scatter(built_lib, world, band):
    env = load("3d_room")
    w, h = 64, 40
    full = env.render((w, h), 0.5, want_hit_ids=True, aovs=ALL)
    for rank in range(world):
        planes = sentinel_planes((h, w), env.dim)
        part = env.render((w, h), 0.5, band_rows=band, band_rank=rank, band_world=world, aovs=planes)
        mine = np.array([(y // band) % world == rank for y in range(h)])
        for n in ALL:
            assert same(part.aovs[n][mine], full.aovs[n][mine]), f"rank {rank}: {n}"
            assert same(part.aovs[n][~mine], sentinel_planes((h, w), env.dim, [n])[n][~mine]), f"rank {rank}: {n} other rows"


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_compact_rows_device_entry(built_lib, pipeline):
    import torch

    env = load("4d_room")
    env.pipeline = pipeline_id(pipeline)
    w, h, world, band = 45, 37, 3, 8
    full = env.render((w, h), 0.0, want_hit_ids=True, aovs=ALL)
    for rank in range(world):
        opts = eb.EuclRenderOpts(width=w, height=h, band_rows=band, band_rank=rank, band_world=world)
        rows = eb.lib().eucl_band_rows_for_rank(C.byref(opts))
        mine = np.array([(y // band) % world == rank for y in range(h)])
        assert mine.sum() == rows
        rgb = torch.zeros((rows, w, 3), dtype=torch.uint8, device="cuda")
        planes = DevicePlanes((int(rows), w), env.dim)
        env.render_device(rgb.data_ptr(), (w, h), 0.0, band_rows=band, band_rank=rank, band_world=world, compact_rows=True,
                          d_aovs=planes.ptrs(ALL))
        assert np.array_equal(rgb.cpu().numpy(), full.data[mine])
        for n in ALL:
            assert same(planes.get(n), full.aovs[n][mine]), f"rank {rank}: {n}"


@pytest.mark.gpu
@pytest.mark.parametrize("split", [2, 3])
@pytest.mark.parametrize("name,size", [("3d_room", (96, 70)), ("4d_room", (80, 53))])
def test_two_pipelines_equal_one(built_lib, monkeypatch, split, name, size):
    monkeypatch.setenv("EUCL_SPLIT_MIN_PIXELS", "0")
    monkeypatch.setenv("EUCL_SPLIT", "1")
    env = load(name)
    one = env.render(size, 0.5, want_hit_ids=True, aovs=ALL)
    monkeypatch.setenv("EUCL_SPLIT", str(split))
    img = check_oracle(env, size, time=0.5)
    assert np.array_equal(img.data, one.data)
    assert_planes(img.aovs, one.aovs)
    assert {k: img.stats[k] for k in COUNTED} == {k: one.stats[k] for k in COUNTED}


@pytest.mark.gpu
def test_forced_arena_retry(built_lib, monkeypatch):
    plain = load("3d_fresnel_2").render((48, 31), want_hit_ids=True, aovs=ALL)
    monkeypatch.setenv("EUCL_ARENA_FACTOR_X10", "11")
    tight = load("3d_fresnel_2").render((48, 31), want_hit_ids=True, aovs=ALL, profile=True)
    assert tight.stats["retries"] > 0
    assert np.array_equal(tight.data, plain.data) and np.array_equal(tight.hit_ids, plain.hit_ids)
    assert_planes(tight.aovs, plain.aovs)


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_pixels", [200, 777])
def test_chunks_end_inside_frames(built_lib, monkeypatch, chunk_pixels):
    monkeypatch.setenv("EUCL_CHUNK_PIXELS", str(chunk_pixels))
    check_oracle(load("3d_room"), (37, 23), time=0.2)


class DevicePlanes:
    """Device planes of every AOV, filled with SENTINEL (uint32 planes held as int32 tensors: the same bytes)."""

    def __init__(self, lead, dim):
        import torch

        self.sentinel = sentinel_planes(lead, dim)
        self.dev = {n: torch.from_numpy(self._raw(a)).cuda() for n, a in self.sentinel.items()}

    @staticmethod
    def _raw(a):
        return a.view(np.int32) if a.dtype == np.uint32 else a

    def refill(self):
        import torch

        for n, t in self.dev.items():
            t.copy_(torch.from_numpy(self._raw(self.sentinel[n])))

    def ptrs(self, names):
        return {n: self.dev[n].data_ptr() for n in names}

    def get(self, n):
        a = self.dev[n].cpu().numpy()
        return a.view(np.uint32) if self.sentinel[n].dtype == np.uint32 else a

    def untouched(self, n):
        return same(self.get(n), self.sentinel[n])


@pytest.mark.gpu
def test_graph_replay_and_alternating_calls(built_lib):
    import torch

    env = load("3d_room")
    w, h = 64, 40
    ref = env.render((w, h), 0.5, want_hit_ids=True, aovs=ALL)
    for _ in range(6):  # the scene settles its ray-grouping mode first (no graphs while it measures)
        env.render((w, h), 0.5)
    rgb = torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda")
    planes = DevicePlanes((h, w), env.dim)
    subset = ["depth", "segments"]
    replays = []
    # three identical AOV calls (direct launch, capture, replay), plain calls, AOVs again, a subset of the planes: every
    # call writes exactly its planes -- a replayed graph of another kind would leave planes stale or write unasked ones
    for step, kind in enumerate(["all"] * 3 + ["plain"] * 3 + ["all", "plain", "subset", "subset", "subset", "all"]):
        rgb.zero_()
        planes.refill()
        names = {"all": ALL, "subset": subset, "plain": []}[kind]
        st = env.render_device(rgb.data_ptr(), (w, h), 0.5, d_aovs=planes.ptrs(names) if names else None)
        replays.append(st["graph_replays"])
        assert np.array_equal(rgb.cpu().numpy(), ref.data), f"step {step}"
        for n in ALL:
            if n in names:
                assert same(planes.get(n), ref.aovs[n]), f"step {step} ({kind}): {n}"
            else:
                assert planes.untouched(n), f"step {step} ({kind}): {n} was written"
    assert replays[:3] == [0, 1, 1] and replays[5] == 1 and replays[10] == 1
    host = env.render((w, h), 0.5, want_hit_ids=True)
    assert host.aovs is None and np.array_equal(host.data, ref.data)


@pytest.mark.gpu
def test_4k_rows_against_oracle(built_lib, monkeypatch):
    monkeypatch.setenv("EUCL_CHUNK_PIXELS", str(3840 * 100))  # chunk boundaries inside the sampled row ranges
    env = load("3d_room")
    w, h = 3840, 2160
    img = env.render((w, h), 0.0, want_hit_ids=True, aovs=ALL)
    assert int(img.aovs["segments"].sum(dtype=np.uint64)) == img.stats["segments"]
    for r0, r1 in [(0, 2), (99, 101), (1599, 1601), (2158, 2160)]:
        rgb, hit, planes, _ = oracle_api.render_aovs(env, w, h, rows=(r0, r1))
        assert np.array_equal(img.data[r0:r1], rgb) and np.array_equal(img.hit_ids[r0:r1], hit)
        assert_planes({n: a[r0:r1] for n, a in img.aovs.items()}, planes, what=f"rows {r0}-{r1}: ")


@pytest.mark.gpu
def test_invalid_arguments_are_rejected(built_lib):
    from euclider_b200._capi import EuclAovs, EuclFrame, EuclRenderOpts, EuclStats

    env = load("3d_room")
    scene = env._device_scene(0)
    lib = eb.lib()
    out = np.zeros((2, 8, 8, 3), np.uint8)
    depth = np.full((2, 8, 8), -7.0, np.float32)

    def call(frames, n, aovs, rgb=out, **opts):
        o = EuclRenderOpts(width=8, height=8, **opts)
        return lib.eucl_render_aovs(scene, frames, n, C.byref(o), rgb.ctypes.data if rgb is not None else None, None,
                                    C.byref(aovs) if aovs is not None else None, C.byref(EuclStats()))

    frames = (EuclFrame * 2)()
    for f in frames:
        f.camera = env.camera.copy()
    good = EuclAovs(depth=depth.ctypes.data)
    for args, kw in [((frames, 2, None), {}), ((frames, 2, EuclAovs()), {}), ((frames, 0, good), {}), ((None, 1, good), {}),
                     ((frames, 2, good), {"band_world": 2, "band_rows": 4}), ((frames, 2, good), {"compact_rows": 1}),
                     ((frames, 2, good), {"rgb": None}), ((frames, 1, good), {"band_world": 2, "band_rank": 2})]:
        assert call(*args, **kw) == EUCL_ERR_INVALID_ARGUMENT, (args, kw)
    assert (depth == -7.0).all()  # rejected before any device work
    assert lib.eucl_render_aovs_device(scene, frames, 1, C.byref(EuclRenderOpts(width=8, height=8)), None, None,
                                       C.byref(good), C.byref(EuclStats())) == EUCL_ERR_INVALID_ARGUMENT
    assert call(frames, 2, good) == 0 and not np.isnan(depth).all()
    # a single frame accepts band-split options
    assert call(frames, 1, good, band_world=2, band_rows=4, band_rank=1) == 0


@pytest.mark.gpu
def test_tool_writes_aov_planes(built_lib, tmp_path):
    scene = ROOT / "assets" / "scenes" / "3d_room.json"
    subprocess.run([sys.executable, str(ROOT / "tools" / "eucl_render.py"), str(scene), str(tmp_path / "f.png"), "--size", "40", "24",
                    "--aov", "depth,normal,segments,levels"], check=True, capture_output=True)
    subprocess.run([sys.executable, str(ROOT / "tools" / "eucl_render.py"), str(scene), str(tmp_path / "s_%04d.png"), "--size", "40",
                    "24", "--frames", "2", "--yaw", "0.1", "--aov", "depth"], check=True, capture_output=True)
    ref = load("3d_room").render((40, 24), aovs=ALL)
    for name in ("depth", "normal", "segments", "levels"):
        assert same(np.load(tmp_path / f"f.{name}.npy"), ref.aovs[name]), name
    for name in ("depth", "segments", "levels"):
        assert (tmp_path / f"f.{name}.png").exists()
    assert not (tmp_path / "f.normal.png").exists()
    assert same(np.load(tmp_path / "s_0000.depth.npy"), ref.aovs["depth"])
    assert (tmp_path / "s_0001.depth.npy").exists() and (tmp_path / "s_0001.depth.png").exists()


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_aovs_struct_layout():
    from euclider_b200._capi import EuclAovs

    assert C.sizeof(EuclAovs) == 40
    assert [getattr(EuclAovs, n).offset for n in ALL] == [0, 8, 16, 24, 32]


@pytest.mark.parametrize("name,size,variant", [("3d_room", (48, 27), "det"), ("4d_room", (40, 23), "det"),
                                               ("3d_fresnel_2", (40, 23), "det"), ("4d_cylinders", (32, 18), "det"),
                                               ("3d_room", (40, 23), "f32"), ("no_void_3d", (24, 16), "det")])
def test_oracle_planes_are_consistent(oracle, name, size, variant):
    env = load(name)
    w, h = size
    rgb, hit, planes, st = oracle_api.render_aovs(env, w, h, time=0.5, variant=variant)
    rgb0, hit0, st0 = oracle.render(env, w, h, time=0.5, variant=variant)
    assert np.array_equal(rgb, rgb0) and np.array_equal(hit, hit0)
    assert st["segments"] == st0["segments"] and st["level_counts"] == st0["level_counts"]
    assert int(planes["segments"].sum(dtype=np.uint64)) == st["segments"]
    lv = planes["levels"]
    assert lv.max() <= env.camera.max_depth + 1 and int(np.bincount(lv.ravel(), minlength=1)[0]) == int((hit == -2).sum())
    hit_mask = hit >= 0
    assert np.isfinite(planes["depth"][hit_mask]).all() and (planes["depth"][hit == -1] == np.inf).all()
    assert np.isnan(planes["depth"][hit == -2]).all() and np.isnan(planes["normal"][~hit_mask]).all()


def test_python_argument_checks():
    env = eb.load_reference_scene("3d_room")
    cam = env.camera.copy()
    with pytest.raises(ValueError):
        env.render((8, 8), aovs=("depth", "albedo"))
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [cam], aovs=["segment"])
    with pytest.raises(ValueError):
        env.render((8, 8), aovs={"depth": np.zeros((8, 8), np.float64)})
    with pytest.raises(ValueError):
        env.render((8, 8), aovs={"position": np.zeros((8, 8, 4), np.float32)})  # 3-D scene: 3 components
    with pytest.raises(ValueError):
        env.render((8, 8), aovs={"segments": np.zeros((8, 8), np.int32)})
    with pytest.raises(ValueError):
        env.render((8, 8), aovs={"levels": np.zeros((16, 8), np.uint32)[::2]})
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [cam, cam], aovs={"depth": np.zeros((8, 8), np.float32)})
    with pytest.raises(ValueError):
        env.render_device(0, (8, 8), d_aovs={"depht": 1234})
    with pytest.raises(ValueError):
        env.render_frames_device(0, (8, 8), [cam], d_aovs={"depth": 0})


def test_tool_aov_option_parsing():
    a = eucl_render.parse_args(["s.json", "out.png"])
    assert a.aov == []
    a = eucl_render.parse_args(["s.json", "out.png", "--aov", "depth,normal,segments,levels"])
    assert a.aov == ["depth", "normal", "segments", "levels"] and not eucl_render.is_sequence(a)
    assert eucl_render.aov_path("out.png", "depth", ".npy") == "out.depth.npy"
    assert eucl_render.aov_path("seq_0003.ppm", "segments", ".png") == "seq_0003.segments.png"
    for bad in (["--aov", "depth,albedo"], ["--aov", ""], ["--aov", "depth,,normal"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o.png", *bad])
