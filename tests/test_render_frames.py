"""Batches of frames (eucl_render_frames*): K frames rendered as one wavefront are, frame by frame, the pictures and hit
maps of K single renders and of the CPU oracle -- bit for bit -- and their summed statistics are the sums of the singles.
The GPU tests cover chunk and band boundaries inside a frame, traced and untraced frames in one batch, both precisions and
pipelines, both entry points, retries and graph replay; the CPU tests cover the ABI struct, argument checks and the
image-sequence options of tools/eucl_render.py."""
import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import eucl_render  # noqa: E402

COUNTED = ("pixels", "segments", "nodes", "level_counts")
EUCL_ERR_INVALID_ARGUMENT = -1


def load(name):
    if name == "no_void_3d":
        return eb.Parser.default(resource_root=ROOT).parse_file(ROOT / "tests" / "scenes" / "no_void_3d.json")
    return eb.load_reference_scene(name)


def camera_path(env, k):
    """k distinct poses: steps through the universe (move_camera) and turns."""
    cams = []
    step = [0.0] * env.dim
    step[1] = 0.15
    step[0] = 0.05
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


def singles(env, size, cams, times, **kw):
    saved = env.camera.copy()
    out = []
    try:
        for cam, t in zip(cams, times):
            env.camera = cam.copy()
            out.append(env.render(size, t, want_hit_ids=True, **kw))
    finally:
        env.camera = saved
    return out


def summed(imgs):
    levels = len(imgs[0].stats["level_counts"])
    return {"pixels": sum(i.stats["pixels"] for i in imgs), "segments": sum(i.stats["segments"] for i in imgs),
            "nodes": sum(i.stats["nodes"] for i in imgs),
            "level_counts": [sum(i.stats["level_counts"][lv] for i in imgs) for lv in range(levels)]}


def assert_batch_equals(batch, ones):
    assert len(batch) == len(ones)
    for k, one in enumerate(ones):
        assert np.array_equal(batch.data[k], one.data), f"frame {k}: pixels differ"
        assert np.array_equal(batch.hit_ids[k], one.hit_ids), f"frame {k}: hit ids differ"
    assert {key: batch.stats[key] for key in COUNTED} == summed(ones)


def check_against_singles_and_oracle(env, oracle, size, cams, times, variant="det"):
    w, h = size
    batch = env.render_frames(size, cams, times, want_hit_ids=True)
    ones = singles(env, size, cams, times)
    assert_batch_equals(batch, ones)
    for k, (cam, t) in enumerate(zip(cams, times)):
        rgb, hit, st = oracle.render(env, w, h, time=t, camera=cam, variant=variant)
        assert np.array_equal(batch.data[k], rgb) and np.array_equal(batch.hit_ids[k], hit), f"frame {k} differs from the oracle"
    return batch


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "3d_fresnel_2", "4d_frame", "3d_hallways"])
def test_batch_equals_singles_and_oracle(built_lib, oracle, name):
    env = load(name)
    cams = camera_path(env, 5)
    times = [0.0, 0.25, 1.5, 1.5004, 7.3]  # distinct Perlin times on 3d_room (the last two: the same whole ms)
    check_against_singles_and_oracle(env, oracle, (37, 23), cams, times)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2, 5])
def test_batch_sizes_odd_frames(built_lib, oracle, k):
    env = load("3d_room")
    cams = camera_path(env, k)
    times = [0.5 + 0.37 * i for i in range(k)]
    check_against_singles_and_oracle(env, oracle, (41, 19), cams, times)


@pytest.mark.gpu
def test_batch_of_one_is_eucl_render(built_lib):
    env = load("4d_room")
    one = env.render((53, 29), 0.75, want_hit_ids=True)
    batch = env.render_frames((53, 29), [env.camera.copy()], [0.75], want_hit_ids=True)
    assert np.array_equal(batch.data[0], one.data) and np.array_equal(batch.hit_ids[0], one.hit_ids)
    for key in COUNTED + ("levels", "launches", "retries"):
        assert batch.stats[key] == one.stats[key], key


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_pixels", [200, 777])
def test_chunks_end_inside_frames(built_lib, oracle, monkeypatch, chunk_pixels):
    monkeypatch.setenv("EUCL_CHUNK_PIXELS", str(chunk_pixels))
    env = load("3d_room")
    cams = camera_path(env, 3)
    check_against_singles_and_oracle(env, oracle, (37, 23), cams, [0.1, 0.2, 0.3])


@pytest.mark.gpu
@pytest.mark.parametrize("split", [2, 3])
@pytest.mark.parametrize("name,size", [("3d_room", (40, 29)), ("4d_room", (33, 45))])
def test_split_pipelines_bands_straddle_frames(built_lib, oracle, monkeypatch, split, name, size):
    monkeypatch.setenv("EUCL_SPLIT", str(split))
    monkeypatch.setenv("EUCL_SPLIT_MIN_PIXELS", "0")
    env = load(name)
    cams = camera_path(env, 4)
    check_against_singles_and_oracle(env, oracle, size, cams, [0.0, 1.0, 2.0, 3.0])


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_traced_and_untraced_frames_mixed(built_lib, oracle, pipeline):
    env = load("no_void_3d")
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL if pipeline == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT
    cams = []
    for loc in [(0, 0, 0), (10, 0, 0), (10.5, 0.5, 0), (0, 0, 0)]:
        cam = env.camera.copy()
        for k in range(3):
            cam.location[k] = loc[k]
        cams.append(cam)
    batch = check_against_singles_and_oracle(env, oracle, (37, 23), cams, [0.0] * 4)
    assert (batch.hit_ids[0] == -2).all() and (batch.hit_ids[3] == -2).all()
    assert (batch.hit_ids[1] != -2).all()
    untraced = env.render_frames((37, 23), [cams[0], cams[3]], want_hit_ids=True)
    assert untraced.stats["segments"] == 0 and untraced.stats["nodes"] == 0 and untraced.stats["pixels"] == 2 * 37 * 23


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_low_precision_and_megakernel(built_lib, oracle, pipeline):
    env = load("3d_room")
    env.precision = "f32"
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL if pipeline == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT
    cams = camera_path(env, 3)
    check_against_singles_and_oracle(env, oracle, (37, 23), cams, [0.2, 0.9, 4.0], variant="f32")


@pytest.mark.gpu
def test_megakernel_f64_batch(built_lib, oracle):
    env = load("4d_frame")
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL
    check_against_singles_and_oracle(env, oracle, (29, 21), camera_path(env, 3), [0.0, 0.0, 0.0])


@pytest.mark.gpu
def test_device_entry_point_with_and_without_hit_ids(built_lib):
    import torch

    env = load("3d_hallways")
    w, h = 45, 27
    cams = camera_path(env, 3)
    host = env.render_frames((w, h), cams, [0.0, 0.5, 1.0], want_hit_ids=True)
    rgb = torch.zeros((3, h, w, 3), dtype=torch.uint8, device="cuda")
    hit = torch.full((3, h, w), -3, dtype=torch.int32, device="cuda")
    st = env.render_frames_device(rgb.data_ptr(), (w, h), cams, [0.0, 0.5, 1.0], d_out_hit_ids=hit.data_ptr())
    assert np.array_equal(rgb.cpu().numpy(), host.data) and np.array_equal(hit.cpu().numpy(), host.hit_ids)
    assert {key: st[key] for key in COUNTED} == {key: host.stats[key] for key in COUNTED}
    rgb2 = torch.zeros_like(rgb)
    env.render_frames_device(rgb2.data_ptr(), (w, h), cams, [0.0, 0.5, 1.0])
    assert torch.equal(rgb2, rgb)
    no_hit = env.render_frames((w, h), cams, [0.0, 0.5, 1.0])
    assert no_hit.hit_ids is None and np.array_equal(no_hit.data, host.data)


@pytest.mark.gpu
def test_retries_give_identical_frames(built_lib, monkeypatch):
    env = load("3d_fresnel_2")
    cams = camera_path(env, 3)
    plain = env.render_frames((48, 31), cams, want_hit_ids=True)
    monkeypatch.setenv("EUCL_ARENA_FACTOR_X10", "11")
    env2 = load("3d_fresnel_2")
    tight = env2.render_frames((48, 31), cams, want_hit_ids=True, profile=True)
    assert tight.stats["retries"] > 0
    assert np.array_equal(tight.data, plain.data) and np.array_equal(tight.hit_ids, plain.hit_ids)
    assert {key: tight.stats[key] for key in COUNTED} == {key: plain.stats[key] for key in COUNTED}


@pytest.mark.gpu
def test_graph_replay_and_changed_frames(built_lib):
    env = load("3d_room")
    size = (64, 40)
    cams = camera_path(env, 4)
    times = [0.0, 0.5, 1.0, 1.5]
    first = env.render_frames(size, cams, times, want_hit_ids=True)
    st = None
    for _ in range(6):
        again = env.render_frames(size, cams, times, want_hit_ids=True)
        assert np.array_equal(again.data, first.data) and np.array_equal(again.hit_ids, first.hit_ids)
        st = again.stats
    assert st["graph_replays"] == 1 and st["retries"] == 0
    # one pose changed: the new picture, not the replayed old one
    moved = [c.copy() for c in cams]
    moved[2].location[0] += 0.3
    changed = env.render_frames(size, moved, times, want_hit_ids=True)
    ref = singles(env, size, moved, times)
    assert_batch_equals(changed, ref)
    assert not np.array_equal(changed.data[2], first.data[2])
    # one time changed (Perlin on 3d_room)
    later = env.render_frames(size, cams, [0.0, 0.5, 1.0, 9.0], want_hit_ids=True)
    assert_batch_equals(later, singles(env, size, cams, [0.0, 0.5, 1.0, 9.0]))
    assert not np.array_equal(later.data[3], first.data[3])


@pytest.mark.gpu
def test_invalid_batches_are_rejected(built_lib):
    from euclider_b200._capi import EuclFrame, EuclRenderOpts, EuclStats

    env = load("3d_room")
    scene = env._device_scene(0)
    lib = eb.lib()
    out = np.zeros((4, 8, 8, 3), np.uint8)

    def call(frames, n, **opts):
        o = EuclRenderOpts(width=8, height=8, **opts)
        return lib.eucl_render_frames(scene, frames, n, C.byref(o), out.ctypes.data, None, C.byref(EuclStats()))

    frames = (EuclFrame * 2)()
    for f in frames:
        f.camera = env.camera.copy()
    assert call(frames, 2) == 0
    assert call(frames, 0) == EUCL_ERR_INVALID_ARGUMENT
    assert call(None, 2) == EUCL_ERR_INVALID_ARGUMENT
    assert call(frames, 2, band_world=2, band_rows=4) == EUCL_ERR_INVALID_ARGUMENT
    assert call(frames, 2, compact_rows=1) == EUCL_ERR_INVALID_ARGUMENT
    frames[1].camera.max_depth = frames[0].camera.max_depth - 1
    assert call(frames, 2) == EUCL_ERR_INVALID_ARGUMENT
    frames[1].camera = env.camera.copy()
    frames[1].camera.dim = 4
    assert call(frames, 2) == EUCL_ERR_INVALID_ARGUMENT
    with pytest.raises(eb.EuclError):
        env.render_frames((8, 8), [env.camera.copy(), frames[1].camera])


@pytest.mark.gpu
def test_tool_writes_an_image_sequence(built_lib, tmp_path):
    scene = ROOT / "assets" / "scenes" / "3d_room.json"
    args = ["--size", "40", "24", "--move", "0.05", "0.2", "0", "--yaw", "0.05", "--time", "0.3", "--time-step", "0.45"]
    subprocess.run([sys.executable, str(ROOT / "tools" / "eucl_render.py"), str(scene), str(tmp_path / "f_%04d.ppm"),
                    "--frames", "4", "--batch", "2", *args], check=True, capture_output=True)
    env = load("3d_room")
    for k in range(4):
        if k:
            env.move_camera([0.05, 0.2, 0.0], 1.0)
            env.rotate_yaw(0.05)
        env.render((40, 24), 0.3 + k * 0.45).save(tmp_path / f"single_{k}.ppm")
        assert (tmp_path / f"f_{k:04d}.ppm").read_bytes() == (tmp_path / f"single_{k}.ppm").read_bytes(), f"frame {k}"


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_frame_struct_layout():
    from euclider_b200._capi import EuclCamera, EuclFrame

    assert C.sizeof(EuclFrame) == 152
    assert EuclFrame.time_seconds.offset == C.sizeof(EuclCamera)


def test_render_frames_checks_its_arguments_before_the_library():
    env = eb.load_reference_scene("3d_room")
    cam = env.camera.copy()
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [cam, cam], times=[0.0])
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [cam], times=[0.0, 1.0])
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [])
    with pytest.raises(ValueError):
        env.render_frames((8, 8), [cam, cam], out=np.zeros((1, 8, 8, 3), np.uint8))
    with pytest.raises(TypeError):
        env.render_frames((8, 8), [(0, 0, 0)])
    with pytest.raises(ValueError):
        env.render_frames_device(0, (8, 8), [cam, cam], times=[0.0, 1.0, 2.0])


def test_tool_argument_parsing():
    a = eucl_render.parse_args(["s.json", "out.png"])
    assert a.frames == 1 and a.batch is None and not eucl_render.is_sequence(a)
    a = eucl_render.parse_args(["s.json", "o_%04d.ppm", "--frames", "4", "--batch", "2", "--move", "0", "0.1", "0",
                                "--yaw", "0.1", "--time-step", "0.5"])
    assert (a.frames, a.batch, a.move, a.yaw, a.time_step) == (4, 2, [0.0, 0.1, 0.0], 0.1, 0.5)
    assert eucl_render.is_sequence(a)
    a = eucl_render.parse_args(["s.json", "o_%04d.ppm", "--frames", "3", "--move", "0", "0", "0", "1",
                                "--plane4", "0", "3", "0.2"])
    assert a.move == [0.0, 0.0, 0.0, 1.0] and a.plane4 == [0.0, 3.0, 0.2]
    for bad in (["--frames", "3"], ["--frames", "0"], ["--batch", "0"], ["--move", "1", "2"],
                ["--plane4", "0.5", "1", "0.1"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o.ppm", *bad])
