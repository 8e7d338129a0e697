"""Scene front end: the reference's JSON constructor vocabulary (src/scene.rs:618-1408) lowered to
flat tables.  Counts per scene follow SURVEY.md App. B."""
import json

import pytest

import euclider_b200 as eb
from euclider_b200 import _capi

# scene -> (dim, surfaced primitives by kind {sphere, plane-like, cylinder}, entities)
EXPECTED = {
    "3d_fresnel": (3, (1, 0, 0), 2),
    "3d_room": (3, (2, 18, 1), 8),
    "3d_hallways": (3, (0, 37, 0), 6),
    "4d_frame": (4, (0, 40, 0), 2),
    "4d_cylinders": (4, (16, 64, 32), 10),
    "4d_room": (4, (3, 24, 1), 8),
}


@pytest.mark.parametrize("name", sorted(EXPECTED))
def test_config_scene_counts(built_lib, name):
    env = eb.load_reference_scene(name)
    flat = env.flat
    dim, (n_sph, n_plane, n_cyl), n_ent = EXPECTED[name]
    assert flat.dim == dim and flat.n_entities == n_ent
    kinds = {1: 0, 2: 0, 3: 0, 4: 0}
    for e in range(flat.n_entities):
        ent = flat.entities[e]
        if ent.surface < 0:
            continue
        for n in range(ent.node_first, ent.node_root + 1):
            if flat.nodes[n].op == _capi.CSG_LEAF:
                k = flat.prims[flat.nodes[n].prim].kind
                if k in kinds:
                    kinds[k] += 1
    assert (kinds[1], kinds[2] + kinds[3], kinds[4]) == (n_sph, n_plane, n_cyl)
    assert env.max_depth() == 10 and env.camera.fov_deg == 90


@pytest.mark.parametrize("name", ["3d_frame", "3d_fresnel_2", "3d_photo", "4d_fresnel"])
def test_other_scenes_parse(built_lib, name):
    env = eb.load_reference_scene(name)
    assert env.flat.n_entities >= 2 and env.flat.n_textures >= 1


def test_post_order_program_layout(built_lib):
    env = eb.load_reference_scene("3d_room")
    flat = env.flat
    for e in range(flat.n_entities):
        ent = flat.entities[e]
        depth = 0
        for n in range(ent.node_first, ent.node_root + 1):
            node = flat.nodes[n]
            if node.op == _capi.CSG_LEAF:
                assert node.first == n
                depth += 1
            else:
                assert flat.nodes[n - 1].first - 1 >= node.first  # `a` subtree ends right before `b` starts
                depth -= 1
        assert depth == 1


def test_cuboid_lowering(built_lib):
    """HalfSpace3::cuboid = left fold of 6 half-spaces with Intersection (d3/entity/shape.rs:17-66)."""
    env = eb.load_reference_scene("3d_room")
    flat = env.flat
    ent = flat.entities[1]  # cuboid c (16, 0, -1) dims (3, 3, 6)
    assert ent.node_root - ent.node_first + 1 == 11
    leaves = [flat.prims[flat.nodes[n].prim] for n in range(ent.node_first, ent.node_root + 1) if flat.nodes[n].op == 0]
    assert [tuple(p.v0[:3]) for p in leaves] == [(1, 0, 0), (1, 0, 0), (0, -1, 0), (0, -1, 0), (0, 0, 1), (0, 0, 1)]
    assert [p.s0 for p in leaves] == [-17.5, -14.5, 1.5, -1.5, -2.0, 4.0]
    assert [p.s1 for p in leaves] == [-1.0, 1.0, 1.0, -1.0, -1.0, 1.0]
    ops = [flat.nodes[n].op for n in range(ent.node_first, ent.node_root + 1)]
    assert ops == [0, 0, 2, 0, 2, 0, 2, 0, 2, 0, 2]


def test_linear_space_expressions(built_lib):
    """3d_hallways: LinearSpace x -> x * 4 (inverse x / 4) compiled to RPN, evaluated per transition."""
    env = eb.load_reference_scene("3d_hallways")
    flat = env.flat
    mats = [flat.materials[flat.entities[e].material] for e in range(flat.n_entities)]
    linear = [m for m in mats if m.kind == _capi.MAT_LINEAR_SPACE]
    assert len(linear) == 2 and all(m.n_transforms == 1 for m in linear)
    t = flat.transforms[linear[0].transform_first]
    ops = [(flat.expr_ops[i].op, flat.expr_ops[i].arg, flat.expr_ops[i].value) for i in range(t.fwd_first[0], t.fwd_first[0] + t.fwd_len[0])]
    assert ops == [(1, 0, 0.0), (0, 0, 4.0), (4, 0, 0.0)]  # VAR x, CONST 4, MUL


def test_json_number_conversion(built_lib):
    """json 0.11 converts (mantissa, exponent) with one multiplication by a power of ten
    (oracle/ASSUMPTIONS.md): 1.458 -> 1458 * 1e-3."""
    env = eb.load_reference_scene("3d_fresnel")
    sf = env.flat.surfaces[0]
    assert sf.ratio_a == 1458 * 1e-3 and sf.ratio_b == 1.0 and sf.thr_a == 1458 * 1e-3


SCENE = {"Universe3": {"camera": {"PitchYawCamera3": []}, "entities": [{"Void3::new_with_vacuum": []}],
                       "background": {"MappedTextureImpl3::new": [{"uv_sphere_3": [{"Point3::new": [0, 0, 0]}]},
                                                                   {"texture_image_linear": ["./x.png"]}]}}}


def parse_error(text):
    with pytest.raises(eb.ParserError) as err:
        eb.Parser.default().parse(text, load_textures=False)
    return err.value.status


def test_parser_errors_mirror_the_reference(built_lib):  # ParserError variants, src/scene.rs:524-552
    assert parse_error("{ not json") == -11  # SyntaxError
    assert parse_error(json.dumps({"NoSuchThing": []})) == -10  # NoDeserializer
    assert parse_error(json.dumps({"a": [], "b": []})) == -13  # InvalidConstructor: single key required
    bad = json.loads(json.dumps(SCENE))
    bad["Universe3"]["camera"] = {"Point3::new": [0, 0, 0]}
    assert parse_error(json.dumps(bad)) == -15  # TypeMismatch
    bad = json.loads(json.dumps(SCENE))
    del bad["Universe3"]["background"]
    assert parse_error(json.dumps(bad)) == -14  # MissingField
    bad = json.loads(json.dumps(SCENE))
    bad["Universe3"]["entities"] = [{"Entity3Impl::new_without_surface": [
        {"Sphere3::new": [{"Point3::new": [0, 0, "x"]}, 1]}, {"Vacuum3::new": []}]}]
    assert parse_error(json.dumps(bad)) == -15


def test_positional_and_keyed_arguments_are_equivalent(built_lib):  # deserializer! macro, src/scene.rs:457-515
    keyed = json.loads(json.dumps(SCENE))
    keyed["Universe3"]["entities"].insert(0, {"Entity3Impl::new_without_surface": {
        "shape": {"Sphere3::new": {"center": {"Point3::new": {"x": 1, "y": 2, "z": 3}}, "radius": 0.5}},
        "material": {"Vacuum3": []}}})
    positional = json.loads(json.dumps(SCENE))
    positional["Universe3"]["entities"].insert(0, {"Entity3Impl::new_without_surface": [
        {"Sphere3": [{"Point3": [1, 2, 3]}, 0.5]}, {"Vacuum3::new": []}]})
    env_a = eb.Parser.default().parse(json.dumps(keyed), load_textures=False)  # keep alive: `flat` borrows
    env_b = eb.Parser.default().parse(json.dumps(positional), load_textures=False)
    a, b = env_a.flat, env_b.flat
    assert tuple(a.prims[0].v0[:3]) == tuple(b.prims[0].v0[:3]) == (1, 2, 3) and a.prims[0].s0 == b.prims[0].s0 == 0.5


def test_reference_construction_panics_become_errors(built_lib):  # shape.rs:750-753, 893-898
    bad = json.loads(json.dumps(SCENE))
    bad["Universe3"]["entities"].insert(0, {"Entity3Impl::new_without_surface": [
        {"Cylinder3::new": [{"Point3": [0, 0, 0]}, {"Vector3": [0, 0, 0]}, 1]}, {"Vacuum3::new": []}]})
    assert parse_error(json.dumps(bad)) == -16
