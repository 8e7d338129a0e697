"""Fresnel / Snell surfaces whose colour program is one constant (3d_room's glass: surface_color_uniform) are shaded by
k_shade_glass, the heavy shade build without the colour-program interpreter (api_device.cu: shade_glass_mask).  Frames,
hit ids, level counts, segments, ray trees and the cost AOVs must equal the oracle and the same scene with the heavy
build (EUCL_SHADE_GLASS=0), in both precisions, through both split pipelines, in batches and across arena retries."""
import json
import re

import numpy as np
import pytest

import euclider_b200 as eb

pytestmark = pytest.mark.gpu

GLASS_SCENES = ["3d_room", "3d_fresnel", "3d_fresnel_2", "3d_photo", "4d_fresnel", "4d_room"]
COUNTED = ("pixels", "segments", "nodes", "level_counts")


def shade_bins(capfd, monkeypatch, render):
    """Runs `render` with EUCL_DUMP_LEVELS=1; returns the (light, glass, heavy) shade masks the dump reports, and the result."""
    monkeypatch.setenv("EUCL_DUMP_LEVELS", "1")
    capfd.readouterr()
    out = render()
    masks = set(re.findall(r"shade bins light (\S+) glass (\S+) heavy (\S+)", capfd.readouterr().err))
    monkeypatch.delenv("EUCL_DUMP_LEVELS")
    assert len(masks) == 1, masks
    return tuple(int(m, 16) for m in masks.pop()), out


def two_pipelines(monkeypatch):
    monkeypatch.setenv("EUCL_SPLIT", "2")
    monkeypatch.setenv("EUCL_SPLIT_MIN_PIXELS", "0")


def reference(name, precision, glass, monkeypatch):
    """A fresh scene with or without k_shade_glass.  The routing is read when the device scene is created, at the first
    render: the caller removes EUCL_SHADE_GLASS after that."""
    monkeypatch.setenv("EUCL_SHADE_GLASS", "1" if glass else "0")
    env = eb.load_reference_scene(name)
    env.precision = precision
    return env


@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("name", GLASS_SCENES)
def test_glass_scenes_equal_oracle_and_heavy_build(built_lib, oracle, capfd, monkeypatch, name, precision):
    two_pipelines(monkeypatch)
    w, h = 160, 90
    rgb, hit, st = oracle.render(eb.load_reference_scene(name), w, h, time=0.5, variant="det" if precision == "f64" else "f32")
    for glass in (True, False):
        env = reference(name, precision, glass, monkeypatch)
        (light, glass_mask, heavy), img = shade_bins(capfd, monkeypatch, lambda: env.render((w, h), time=0.5, want_hit_ids=True))
        monkeypatch.delenv("EUCL_SHADE_GLASS")
        if not glass:
            assert glass_mask == 0
        elif name == "3d_room":
            assert glass_mask != 0 and heavy == 0  # both glass entities have a one-constant colour program
        for k in range(4):  # the ray-grouping tuner, then a captured graph and its replays
            if k:
                img = env.render((w, h), time=0.5, want_hit_ids=True)
            assert np.array_equal(img.data, rgb), (glass, k)
            assert np.array_equal(img.hit_ids, hit), (glass, k)
            assert img.stats["level_counts"] == st["level_counts"], (glass, k)
            assert img.stats["segments"] == st["segments"], (glass, k)


def camera_path(env, k):
    """k distinct poses: steps through the universe and turns."""
    cams = [env.camera.copy()]
    for _ in range(k - 1):
        env.move_camera([0.05, 0.15] + [0.0] * (env.dim - 2), 1.0)
        if env.dim == 3:
            env.rotate_yaw(0.07)
        else:
            env.rotate_plane4(0, 1, 0.06)
        cams.append(env.camera.copy())
    return cams


@pytest.mark.parametrize("name", ["3d_room", "4d_fresnel"])
def test_batch_equals_sequential_renders(built_lib, name):
    env = eb.load_reference_scene(name)
    cams, times = camera_path(env, 3), [0.0, 0.75, 2.5]
    batch = env.render_frames((64, 40), cams, times, want_hit_ids=True)
    for k, (cam, t) in enumerate(zip(cams, times)):
        env.camera = cam.copy()
        one = env.render((64, 40), t, want_hit_ids=True)
        assert np.array_equal(batch.data[k], one.data) and np.array_equal(batch.hit_ids[k], one.hit_ids), k


@pytest.mark.parametrize("name", ["3d_room", "4d_fresnel"])
def test_ray_trees_through_glass(built_lib, oracle, name):
    env = eb.load_reference_scene(name)
    w, h = 96, 54
    pixels = [(x, y) for y in range(0, h, 9) for x in range(0, w, 8)]
    got = env.render((w, h), want_hit_ids=True, trees=pixels)
    want = oracle.pixel_trees(env, w, h, pixels)
    for p, a, b in zip(pixels, got.trees, want):
        assert oracle.first_difference(a, b) is None, p
    # the sampled pixels do reach glass: some node has both a transmitted and a reflected child
    assert any(((t.nodes["level"] == 1).sum() >= 2) for t in got.trees)


@pytest.mark.parametrize("name", ["3d_room", "4d_fresnel"])
def test_cost_aovs_unchanged(built_lib, monkeypatch, name):
    planes = []
    for glass in (True, False):
        env = reference(name, "f64", glass, monkeypatch)
        img = env.render((80, 45), 0.5, want_hit_ids=True, aovs=["segments", "levels"])
        monkeypatch.delenv("EUCL_SHADE_GLASS")
        assert int(img.aovs["segments"].sum(dtype=np.uint64)) == img.stats["segments"]
        planes.append(img.aovs)
    for n in ("segments", "levels"):
        assert np.array_equal(planes[0][n], planes[1][n]), n


def lit_glass_scene():
    """A Fresnel / Snell sphere whose colour program blends two providers, next to one with a constant colour."""
    def P(xs):
        return {"Point3::new": [float(v) for v in xs]}

    def glass(color):
        return {"ComposableSurface3": {
            "reflection_ratio": {"reflection_ratio_fresnel_3": [1.458, 1.0]},
            "reflection_direction": {"reflection_direction_specular_3": []},
            "threshold_direction": {"threshold_direction_snell_3": [1.458]},
            "surface_color": color}}

    lit = {"surface_color_blend_3": [
        {"surface_color_illumination_global_3": [{"Rgba::new": [1, 1, 1, 0]}, {"Rgba::new": [0, 0, 0, 0.6]}]},
        {"surface_color_uniform_3": [{"Rgba::new": [0.2, 0.4, 0.9, 0.3]}]},
        {"blend_function_darken": []}]}
    plain = {"surface_color_uniform_3": [{"Rgba::new": [0, 0, 0, 0.1]}]}
    wall = {"ComposableSurface3": {
        "reflection_ratio": {"reflection_ratio_uniform_3": [0.3]},
        "reflection_direction": {"reflection_direction_specular_3": []},
        "threshold_direction": {"threshold_direction_identity_3": []},
        "surface_color": {"surface_color_illumination_global_3": [{"Rgba::new": [1, 1, 1, 1]}, {"Rgba::new": [0.1, 0.1, 0.1, 1]}]}}}
    entity = lambda shape, surface: {"Entity3Impl::new": [shape, {"Vacuum3::new": []}, surface]}
    room = {"ComposableShape3::of": [[{"VoidShape3": []}, {"HalfSpace3::cuboid": [P([3, 0, 0]), {"Vector3::new": [30.0, 16.0, 9.0]}]}],
                                    {"SetOperation": ["Complement"]}]}
    return json.dumps({"Universe3": {
        "camera": {"PitchYawCamera3::new_with_location": [P([-4.0, 0.3, 0.2])]},
        "entities": [entity({"Sphere3::new": [P([6, -1.5, 0]), 2.5]}, glass(lit)),
                     entity({"Sphere3::new": [P([6, 2.5, 0.5]), 1.5]}, glass(plain)),
                     entity(room, wall), {"Void3::new_with_vacuum": []}],
        "background": {"MappedTextureImpl3::new": [{"uv_sphere_3": [P([0, 0, 0])]}, {"texture_image_linear": ["./t.png"]}]}}})


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_glass_with_a_colour_program_keeps_the_heavy_build(built_lib, oracle, capfd, monkeypatch, precision):
    two_pipelines(monkeypatch)
    env = eb.Parser.default().parse(lit_glass_scene(), load_textures=False)
    env.set_texture(0, 2, 2, bytes([255, 0, 0, 255, 0, 255, 0, 255, 0, 0, 255, 255, 255, 255, 255, 255]))
    env.precision = precision
    w, h = 120, 68
    rgb, hit, st = oracle.render(env, w, h, variant="det" if precision == "f64" else "f32")
    (light, glass, heavy), img = shade_bins(capfd, monkeypatch, lambda: env.render((w, h), want_hit_ids=True))
    # one entity's bins each: the blended-colour sphere on the heavy build, the constant-colour one on k_shade_glass
    assert bin(heavy).count("1") == 3 and bin(glass).count("1") == 3 and light & (heavy | glass) == 0
    for k in range(3):
        if k:
            img = env.render((w, h), want_hit_ids=True)
        assert np.array_equal(img.data, rgb) and np.array_equal(img.hit_ids, hit), k
        assert img.stats["level_counts"] == st["level_counts"], k


def test_arena_retry_renders_the_same_frame(built_lib, monkeypatch):
    plain = eb.load_reference_scene("3d_room").render((64, 36), want_hit_ids=True)
    monkeypatch.setenv("EUCL_ARENA_FACTOR_X10", "11")
    got = eb.load_reference_scene("3d_room").render((64, 36), want_hit_ids=True, profile=True)
    assert got.stats["retries"] > 0
    assert np.array_equal(got.data, plain.data) and np.array_equal(got.hit_ids, plain.hit_ids)
    assert {k: got.stats[k] for k in COUNTED} == {k: plain.stats[k] for k in COUNTED}


@pytest.mark.parametrize("name", ["3d_hallways", "4d_frame", "4d_cylinders"])
def test_scenes_without_glass_launch_no_glass_kernel(built_lib, capfd, monkeypatch, name):
    env = eb.load_reference_scene(name)
    (light, glass, heavy), _ = shade_bins(capfd, monkeypatch, lambda: env.render((64, 36)))
    assert glass == 0
