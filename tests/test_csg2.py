"""Two-leaf CSG entities -- M_OP(op, A, B) with A a primitive or a chain of at most kPlaneChainMax half-spaces and B a
primitive, like 3d_room's glass Complement(cuboid, sphere) -- are evaluated in registers by csg2_first, and a scene whose
surfaced entities are all primitives, root plane chains or such programs walks its heavy rays with k_intersect_csg2
(api_device.cu: ENT_CSG2, SceneHeader::csg2_capable).  Frames, hit ids and level counts must equal the oracle bit for bit
and the same scene with the general heavy build (EUCL_CSG2=0), in both precisions and both dimensions."""
import json
import re

import numpy as np
import pytest

import euclider_b200 as eb

pytestmark = pytest.mark.gpu

OPS = ["Union", "Intersection", "Complement", "SymmetricDifference"]
A_KINDS = ["sphere", "cylinder", "cuboid", "union_planes"]
CENTRE = [6.0, 0.0, 0.0, 0.0]
INSIDE_SHAPE = [3.2, 0.3, 0.2, 0.1]       # inside A (every A kind) and outside B
INSIDE_SUBTRACTED = [6.8, 0.2, 0.1, 0.05]  # inside B, the operand a Complement subtracts


def P(d, xs):
    return {f"Point{d}::new": [float(v) for v in list(xs)[:d]]}


def V(d, xs):
    return {f"Vector{d}::new": [float(v) for v in list(xs)[:d]]}


def OF(d, shapes, op):
    return {f"ComposableShape{d}::of": [shapes, {"SetOperation": [op]}]}


def box(d, c, dims):
    return {"HalfSpace3::cuboid": [P(d, c), V(d, dims)]} if d == 3 else {"HalfSpace4::hypercuboid": [P(d, c), V(d, dims)]}


def half_space(d, normal, through, inside):
    return {f"HalfSpace{d}::new_with_point": [{f"Hyperplane{d}::new_with_point": [V(d, normal), P(d, through)]}, P(d, inside)]}


def shape(d, kind, c=CENTRE):
    c = np.asarray(c, dtype=float)
    if kind == "sphere":
        return {f"Sphere{d}::new": [P(d, c), 3.4]}
    if kind == "small_sphere":
        return {f"Sphere{d}::new": [P(d, c + [0.8, 0, 0, 0]), 1.6]}
    if kind == "cylinder":  # axis exactly along z: rays along z give a = 0, infinite and NaN roots
        return {f"Cylinder{d}::new": [P(d, c), V(d, [0, 0, 1, 0]), 3.3]}
    if kind == "small_cylinder":
        return {f"Cylinder{d}::new": [P(d, c + [0.8, 0, 0, 0]), V(d, [0, 0, 1, 0]), 1.5]}
    if kind == "cuboid":  # a plane chain (Intersection)
        return box(d, c, [6.0, 5.0, 4.0, 4.0])
    if kind == "union_planes":  # a Union chain of half-spaces: everything but a corner
        return OF(d, [half_space(d, [1, 0, 0, 0], c + [2.0, 0, 0, 0], c + [3.0, 0, 0, 0]),
                      half_space(d, [0, 1, 0, 0], c + [0, 1.5, 0, 0], c + [0, 2.5, 0, 0]),
                      half_space(d, [0, 0, -1, 0], c + [0, 0, -1.2, 0], c + [0, 0, -2.0, 0])], "Union")
    if kind == "capped_cylinder":  # a chain that is not made of half-spaces only
        return {f"Cylinder{d}::new_with_height": [P(d, c), V(d, [0, 0, 1, 0]), 3.0, 4.0]}
    raise ValueError(kind)


def surface(d, glass):
    if glass:
        return {f"ComposableSurface{d}": {
            "reflection_ratio": {f"reflection_ratio_fresnel_{d}": [1.458, 1.0]},
            "reflection_direction": {f"reflection_direction_specular_{d}": []},
            "threshold_direction": {f"threshold_direction_snell_{d}": [1.458]},
            "surface_color": {f"surface_color_uniform_{d}": [{"Rgba::new": [0, 0, 0, 0.1]}]}}}
    lit = {f"surface_color_blend_{d}": [
        {f"surface_color_illumination_global_{d}": [{"Rgba::new": [1, 1, 1, 0]}, {"Rgba::new": [0, 0, 0, 0.6]}]},
        {f"surface_color_illumination_directional_{d}": [V(d, [0.3, 0.2, -1, 0.1]), {"Rgba::new": [0.3, 0.5, 1, 1]},
                                                         {"Rgba::new": [0.1, 0.1, 0.1, 1]}]},
        {"blend_function_darken": []}]}
    return {f"ComposableSurface{d}": {
        "reflection_ratio": {f"reflection_ratio_uniform_{d}": [0.3]},
        "reflection_direction": {f"reflection_direction_specular_{d}": []},
        "threshold_direction": {f"threshold_direction_identity_{d}": []}, "surface_color": lit}}


def scene(d, csg, camera=(-4.0, 0.3, 0.2, 0.1), room=None):
    """`csg` as the glass entity in front of the camera, a small opaque sphere, and a room around everything: by default
    Complement(VoidShape, box) (a negated room), or `room` as that room's interior."""
    entity = lambda s, glass: {f"Entity{d}Impl::new": [s, {f"Vacuum{d}::new": []}, surface(d, glass)]}
    interior = room if room is not None else box(d, [3, 0, 0, 0], [30, 16, 9, 9])
    uv = {"uv_sphere_3": [{"Point3::new": [0, 0, 0]}]}
    cam = ({"PitchYawCamera3::new_with_location": [P(d, camera)]} if d == 3 else
           {"FreeCamera4::new_with_location": [P(d, camera)]})
    return json.dumps({f"Universe{d}": {"camera": cam, "entities": [
        entity(csg, True),
        entity({f"Sphere{d}::new": [P(d, [5, -3, 1.5, 0.5]), 1.0]}, False),
        entity(OF(d, [{f"VoidShape{d}": []}, interior], "Complement"), False),
        {f"Void{d}::new_with_vacuum": []}],
        "background": {f"MappedTextureImpl{d}::new": [uv if d == 3 else {"uv_derank_4": [uv]},
                                                      {"texture_image_linear": ["./t.png"]}]}}})


def load(text, precision):
    env = eb.Parser.default().parse(text, load_textures=False)
    env.set_texture(0, 2, 2, bytes([255, 0, 0, 255, 0, 255, 0, 255, 0, 0, 255, 255, 255, 255, 255, 255]))
    env.precision = precision
    return env


def csg2_capable(capfd, monkeypatch, render):
    """Runs `render` with EUCL_DUMP_LEVELS=1 and returns the scene's csg2_capable as the per-chunk dump reports it."""
    monkeypatch.setenv("EUCL_DUMP_LEVELS", "1")
    capfd.readouterr()
    out = render()
    flags = {int(v) for v in re.findall(r"csg2_capable (\d)", capfd.readouterr().err)}
    monkeypatch.delenv("EUCL_DUMP_LEVELS")
    assert len(flags) == 1, flags
    return flags.pop(), out


def check_frames(oracle, capfd, monkeypatch, text, expect_csg2=True, size=(96, 54)):
    """Every frame of the default build and of EUCL_CSG2=0 against the oracle, f64 and f32.  Five frames each way: the
    ray-grouping tuner renders with and without reach-key lists, then a graph is captured and replayed."""
    w, h = size
    for precision, variant in (("f64", "det"), ("f32", "f32")):
        env = load(text, precision)
        rgb, hit, st = oracle.render(env, w, h, variant=variant)
        for csg2 in (True, False):
            if not csg2:
                monkeypatch.setenv("EUCL_CSG2", "0")  # read at eucl_scene_create: a fresh scene
                env = load(text, precision)
            flag, img = csg2_capable(capfd, monkeypatch, lambda: env.render((w, h), want_hit_ids=True))
            assert flag == (1 if csg2 and expect_csg2 else 0)
            for k in range(5):
                if k:
                    img = env.render((w, h), want_hit_ids=True)
                assert np.array_equal(img.hit_ids, hit), (precision, csg2, k)
                assert np.array_equal(img.data, rgb), (precision, csg2, k)
                assert img.stats["level_counts"] == st["level_counts"], (precision, csg2, k)
            monkeypatch.delenv("EUCL_CSG2", raising=False)


def two_leaf(op, a_kind):
    """Whether OF([A, B], op) stays a two-leaf program: a Union / Intersection over a primitive A, or over a chain A of
    the same operation, folds into one chain of leaves that are not all half-spaces (api_device.cu: MacroBuilder)."""
    if op in ("Union", "Intersection") and a_kind in ("sphere", "cylinder"):
        return False
    return (op, a_kind) not in (("Intersection", "cuboid"), ("Union", "union_planes"))


@pytest.mark.parametrize("b_kind", ["small_sphere", "small_cylinder"])
@pytest.mark.parametrize("a_kind", A_KINDS)
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dim", [3, 4])
def test_two_leaf_programs(built_lib, oracle, capfd, monkeypatch, dim, op, a_kind, b_kind):
    check_frames(oracle, capfd, monkeypatch, scene(dim, OF(dim, [shape(dim, a_kind), shape(dim, b_kind)], op)),
                 expect_csg2=two_leaf(op, a_kind))


@pytest.mark.parametrize("where", ["inside_shape", "inside_subtracted"])
@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dim", [3, 4])
def test_cameras_inside_the_operands(built_lib, oracle, capfd, monkeypatch, dim, op, where):
    camera = INSIDE_SHAPE if where == "inside_shape" else INSIDE_SUBTRACTED
    for a_kind in ("cuboid", "sphere"):
        check_frames(oracle, capfd, monkeypatch,
                     scene(dim, OF(dim, [shape(dim, a_kind), shape(dim, "small_sphere")], op), camera=camera),
                     expect_csg2=two_leaf(op, a_kind))


@pytest.mark.parametrize("dim", [3, 4])
def test_negated_two_leaf_room(built_lib, oracle, capfd, monkeypatch, dim):
    """A room whose interior is a two-leaf program: ENT_CSG2 and ENT_NEGATED on one entity."""
    interior = OF(dim, [box(dim, [3, 0, 0, 0], [30, 16, 9, 9]), {f"Sphere{dim}::new": [P(dim, [12, 0, 0, 0]), 5.0]}], "Complement")
    check_frames(oracle, capfd, monkeypatch, scene(dim, shape(dim, "sphere"), room=interior))


@pytest.mark.parametrize("kind", ["non_plane_chain_a", "chain_b", "three_levels"])
@pytest.mark.parametrize("dim", [3, 4])
def test_other_programs_keep_the_general_build(built_lib, oracle, capfd, monkeypatch, dim, kind):
    """Programs csg2_first does not take: the scene runs the general heavy build, with or without EUCL_CSG2."""
    if kind == "non_plane_chain_a":
        csg = OF(dim, [shape(dim, "capped_cylinder"), shape(dim, "small_sphere")], "Complement")
    elif kind == "chain_b":
        csg = OF(dim, [shape(dim, "sphere"), box(dim, [6.8, 0, 0, 0], [2, 2, 2, 2])], "Complement")
    else:
        csg = OF(dim, [shape(dim, "cuboid"), OF(dim, [shape(dim, "small_sphere"), shape(dim, "small_cylinder")], "SymmetricDifference")],
                 "Complement")
    check_frames(oracle, capfd, monkeypatch, scene(dim, csg), expect_csg2=False)


def axis_rays(dim):
    """Axis-parallel rays from points on the faces, edges and centre of the cuboid operand and from inside the sphere:
    parallel planes give infinite and NaN distances, head-on hits on the Snell glass give NaN child directions."""
    c = np.asarray(CENTRE[:dim])
    half = np.asarray([3.0, 2.5, 2.0, 2.0][:dim])
    starts = [c, c + np.eye(dim)[0] * 0.8, np.asarray([0.0, 0.3, 0.2, 0.1][:dim])]
    for k in range(dim):
        for s in (-1.0, 1.0):
            p = c.copy()
            p[k] += s * half[k]
            starts.append(p)
            q = p.copy()
            q[(k + 1) % dim] += half[(k + 1) % dim]  # on an edge
            starts.append(q)
    dirs = []
    for k in range(dim):
        for s in (-1.0, 1.0):
            e = np.zeros(dim)
            e[k] = s
            dirs.append(e)
    o = np.repeat(np.asarray(starts), len(dirs), axis=0)
    d = np.tile(np.asarray(dirs), (len(starts), 1))
    return o, d


@pytest.mark.parametrize("op", OPS)
@pytest.mark.parametrize("dim", [3, 4])
def test_axis_parallel_rays(built_lib, oracle, monkeypatch, dim, op):
    text = scene(dim, OF(dim, [shape(dim, "cuboid"), shape(dim, "small_cylinder")], op))
    o, d = axis_rays(dim)
    for precision, variant in (("f64", "det"), ("f32", "f32")):
        env = load(text, precision)
        rgb, hit, _, st = oracle.trace_rays(env, o, d, variant=variant)
        got = [env.trace_rays(o, d) for _ in range(3)]
        monkeypatch.setenv("EUCL_CSG2", "0")
        got.append(load(text, precision).trace_rays(o, d))
        monkeypatch.delenv("EUCL_CSG2")
        for g in got:
            assert np.array_equal(g.data, rgb) and np.array_equal(g.hit_ids, hit), precision
            assert g.stats["level_counts"] == st["level_counts"], precision
    # the rays do reach the degenerate cases: some child direction is NaN
    env = load(text, "f64")
    trees = [oracle.ray_tree(env, o[i], d[i]) for i in range(len(o))]
    assert any(np.isnan(t.nodes["direction"][:, :dim]).any() for t in trees)


@pytest.mark.parametrize("precision", ["f64", "f32"])
def test_3d_room_takes_the_csg2_build(built_lib, oracle, capfd, monkeypatch, precision):
    env = eb.load_reference_scene("3d_room")
    env.precision = precision
    w, h = 192, 108
    rgb, hit, st = oracle.render(env, w, h, variant="det" if precision == "f64" else "f32")
    flag, img = csg2_capable(capfd, monkeypatch, lambda: env.render((w, h), want_hit_ids=True))
    assert flag == 1
    assert np.array_equal(img.data, rgb) and np.array_equal(img.hit_ids, hit)
    assert img.stats["level_counts"] == st["level_counts"]
    monkeypatch.setenv("EUCL_CSG2", "0")
    env0 = eb.load_reference_scene("3d_room")
    env0.precision = precision
    flag0, img0 = csg2_capable(capfd, monkeypatch, lambda: env0.render((w, h), want_hit_ids=True))
    assert flag0 == 0
    assert np.array_equal(img0.data, rgb) and np.array_equal(img0.hit_ids, hit)


@pytest.mark.parametrize("name", ["3d_hallways", "4d_frame", "4d_cylinders"])
def test_other_reference_scenes_keep_todays_kernels(built_lib, capfd, monkeypatch, name):
    """Their programs have chains on both sides or more than two operands: not csg2-capable."""
    env = eb.load_reference_scene(name)
    flag, _ = csg2_capable(capfd, monkeypatch, lambda: env.render((64, 36)))
    assert flag == 0
