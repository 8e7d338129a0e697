"""Universe::trace_path_unknown (src/universe/mod.rs:186-227,273-286; surface.rs:164-197): the step
before the hot path (camera translation through voids).  Oracle semantics on the CPU; CUDA kernel vs
oracle bit for bit on the GPU."""
import numpy as np
import pytest

import euclider_b200 as eb


def test_straight_line_in_vacuum(oracle, built_lib):
    env = eb.load_reference_scene("3d_fresnel")  # sphere c (10,0,0) r 3 in a vacuum void
    loc, d = oracle.trace_path(env, (0, 0, 0), (0, 1, 0), 2.5)
    assert loc == [0.0, 2.5, 0.0] and d == [0.0, 1.0, 0.0]
    # through the glass sphere: surfaces are crossed, Vacuum materials do not bend or stretch the path
    loc, d = oracle.trace_path(env, (0, 0, 0), (1, 0, 0), 20.0)
    assert d == [1.0, 0.0, 0.0]
    assert loc[0] == pytest.approx(20.0 + 2 * 1.28e-4, abs=1e-9) and loc[1:] == [0.0, 0.0]  # two self-hit offsets


def test_linear_space_void_stretches_the_step(oracle, built_lib):
    """3d_hallways entity 0: cuboid c (20,-5,-1) dims (20,3,6) whose LinearSpace maps x -> 4x: a step of
    length L along +x inside it covers 4L; leaving the void restores the direction (inverse x / 4)."""
    env = eb.load_reference_scene("3d_hallways")
    start = (12.0, -5.0, -1.0)  # inside the stretching hallway (x in [10, 30])
    loc, d = oracle.trace_path(env, start, (1, 0, 0), 1.0)
    assert loc == [16.0, -5.0, -1.0] and d == [1.0, 0.0, 0.0]
    # from outside, walking in: 3 units to the portal at x = 10, the remaining 2 are stretched to 8
    loc, d = oracle.trace_path(env, (7.0, -5.0, -1.0), (1, 0, 0), 5.0)
    assert loc[0] == pytest.approx(10.0 + 8.0, abs=1e-2) and d == [1.0, 0.0, 0.0]


def test_none_outside_every_entity(oracle, built_lib):
    from test_oracle_semantics import SPH, scene_with  # a scene whose only non-void entity is a sphere...

    env = scene_with([SPH((0, 0, 0), 1)])
    assert oracle.trace_path(env, (5, 0, 0), (1, 0, 0), 1.0) is not None  # the Void entity contains everything


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_hallways", "3d_room", "4d_room", "3d_fresnel", "4d_cylinders"])
def test_gpu_matches_oracle(oracle, built_lib, name):
    env = eb.load_reference_scene(name)
    rng = np.random.default_rng(7)
    dim = env.dim
    for _ in range(60):
        loc = rng.uniform(-8, 28, dim)
        loc[2] = rng.uniform(-3.5, 5.0)
        d = rng.normal(size=dim)
        d /= np.linalg.norm(d)
        dist = float(rng.uniform(0.1, 60.0))
        want = oracle.trace_path(env, loc, d, dist)
        got = env.trace_path_unknown(loc, d, dist)
        assert (want is None) == (got is None)
        if want is not None:
            assert got[0] == want[0] and got[1] == want[1]  # bit-exact


@pytest.mark.gpu
def test_move_camera_changes_the_frame(built_lib, oracle):
    env = eb.load_reference_scene("3d_hallways")
    before = env.render((96, 54)).data.copy()
    assert env.move_camera((1, 0, 0), 4.0)
    assert env.camera.location[0] == 4.0
    rgb, _, _ = oracle.render(env, 96, 54)
    after = env.render((96, 54)).data
    assert np.array_equal(after, rgb) and not np.array_equal(after, before)
