"""Ray-tree inspection (eucl_render_trees, eucl_trace_ray_trees; Environment.render / render_frames / trace_rays with
`trees=`): the trees equal the CPU oracle's restatement of Tracer::trace (oracle/oracle_features.cc) node for node and bit for
bit, any NaN equal to any NaN, for both pipelines and both precisions; a tree call renders exactly what the plain call
renders; every tree agrees with the pixel, the hit id and the AOV planes; and the trees survive the frame machinery (chunks,
split pipelines, arena retries, duplicate items, graph replays around them).  The CPU tests pin the ABI layout, the Python
argument checks, the tool's --inspect option and the oracle restatement against oracle.cc itself."""
import ctypes as C
import json
import math
import shutil
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb
import oracle_api
from euclider_b200 import _capi

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "tools"))
import eucl_render  # noqa: E402

ALL = eb.AOV_NAMES
SCENES = sorted(p.stem for p in (ROOT / "assets" / "scenes").glob("*.json"))
COUNTED = ("pixels", "segments", "nodes", "level_counts")
EUCL_OK, EUCL_ERR_INVALID_ARGUMENT = 0, -1


def load(name):
    if name in ("no_void_3d", "csg_mix_3d"):  # csg_mix_3d holds a LinearSpace void
        return eb.Parser.default(resource_root=ROOT).parse_file(ROOT / "tests" / "scenes" / f"{name}.json")
    return eb.load_reference_scene(name)


def pipeline_id(name):
    return eb.EUCL_PIPELINE_MEGAKERNEL if name == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT


def same(a, b) -> bool:
    """Equal values, except that any NaN equals any NaN."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na], b[~nb])


def counted(stats):
    return {k: stats[k] for k in COUNTED}


def assert_trees_equal(got, want, labels):
    assert len(got) == len(want) == len(labels)
    for label, a, b in zip(labels, got, want):
        diff = oracle_api.first_difference(a, b)
        assert diff is None, f"item {label}: {diff}"


def check_consistency(env, trees, cells, rgb, hit, planes, max_depth):
    """Each tree against the other outputs of its item (`cells`: indices into rgb / hit / the planes): the composited root
    is the pixel, the root hit the hit id, the root t and normal the depth and normal planes after narrowing, and the
    node levels give segments and levels."""
    variant = oracle_api.variant_of(env)
    for cell, tr in zip(cells, trees):
        root = tr.nodes[0]
        checker = bool(root["flags"] & _capi.EUCL_TREE_CHECKERBOARD)
        assert root["parent"] == -1 and root["level"] == 0 and root["kind"] == _capi.EUCL_TREE_ROOT
        assert np.array_equal(oracle_api.tree_pixel(root, variant), rgb[cell]), (cell, tr.format())
        assert (-2 if checker else root["hit_entity"]) == hit[cell], cell
        with np.errstate(over="ignore"):  # narrowing, as the depth plane does
            assert same(np.float32(root["t"]), planes["depth"][cell]), cell
        assert same(root["normal"][:env.dim].astype(np.float32), planes["normal"][cell]), cell
        if not tr.truncated:
            levels = tr.nodes["level"]
            assert (0 if checker else int((levels < max_depth).sum())) == planes["segments"][cell], cell
            assert (0 if checker else int(levels.max()) + 1) == planes["levels"][cell], cell
            assert tr.count == len(tr.nodes)


def sample_pixels(w, h, seed, segments=None, n=64):
    """Seeded random pixels, the corners, the centre and the pixel with the most segments."""
    rng = np.random.default_rng(seed)
    px = [(int(x), int(y)) for x, y in zip(rng.integers(0, w, n), rng.integers(0, h, n))]
    px += [(0, 0), (w - 1, 0), (0, h - 1), (w - 1, h - 1), (w // 2, h // 2)]
    if segments is not None:
        y, x = np.unravel_index(int(np.argmax(segments)), segments.shape)
        px.append((int(x), int(y)))
    return px


def check_render_trees(env, size, time=0.0, pixels=None, capacity=None, seed=0):
    """A camera tree call against the plain call, the AOV planes and the oracle."""
    w, h = size
    md = int(env.camera.max_depth)
    plain = env.render(size, time, want_hit_ids=True, aovs=ALL)
    if pixels is None:
        pixels = sample_pixels(w, h, seed, plain.aovs["segments"])
    got = env.render(size, time, want_hit_ids=True, trees=pixels, tree_capacity=capacity)
    assert np.array_equal(got.data, plain.data) and np.array_equal(got.hit_ids, plain.hit_ids)
    assert counted(got.stats) == counted(plain.stats)
    assert len(got.trees) == len(pixels)
    check_consistency(env, got.trees, [(y, x) for x, y in pixels], plain.data, plain.hit_ids, plain.aovs, md)
    cap = eb.default_tree_capacity(md) if capacity is None else capacity
    want = oracle_api.pixel_trees(env, w, h, pixels, time, capacity=cap)
    assert_trees_equal(got.trees, want, pixels)
    return got


def scene_extent(env) -> float:
    flat, dim = env.flat, env.dim
    ext = max(10.0, float(np.linalg.norm([env.camera.location[k] for k in range(dim)])))
    for i in range(flat.n_prims):
        p = flat.prims[i]
        if p.kind == 1 and math.isfinite(p.s0):
            ext = max(ext, float(np.linalg.norm([p.v0[k] for k in range(dim)])) + abs(p.s0))
    return ext


def random_rays(env, n, seed):
    """Half the origins near the camera, half spread over and beyond the scene; unnormalised random directions."""
    rng = np.random.default_rng(seed)
    dim, ext = env.dim, scene_extent(env)
    loc = np.array([env.camera.location[k] for k in range(dim)])
    origins = np.concatenate([loc + rng.normal(0.0, 0.05 * ext, (n // 2, dim)), rng.uniform(-1.5 * ext, 1.5 * ext, (n - n // 2, dim))])
    d = rng.normal(size=(n, dim))
    d *= (10.0 ** rng.uniform(-3, 3, (n, 1))) / np.linalg.norm(d, axis=1, keepdims=True)
    return origins, d


def check_ray_trees(env, o, d, items, time=0.0, max_depth=None, width=None, capacity=None):
    """A ray tree call against the plain call, the AOV planes and the oracle.  `items`: flat indices or index tuples."""
    md = int(env.camera.max_depth if max_depth is None else max_depth)
    plain = env.trace_rays(o, d, time, max_depth=max_depth, width=width, aovs=ALL)
    got = env.trace_rays(o, d, time, max_depth=max_depth, width=width, trees=items, tree_capacity=capacity)
    assert np.array_equal(got.data, plain.data) and np.array_equal(got.hit_ids, plain.hit_ids)
    assert counted(got.stats) == counted(plain.stats)
    lead = o.shape[:-1]
    flat = [int(np.ravel_multi_index(i, lead)) if isinstance(i, tuple) else int(i) for i in items]
    cells = [np.unravel_index(i, lead) for i in flat]
    check_consistency(env, got.trees, cells, plain.data, plain.hit_ids, plain.aovs, md)
    w = width if width is not None else (lead[-1] if len(lead) >= 2 else 1)
    w = max(int(w), 1)
    of, df = o.reshape(-1, env.dim), d.reshape(-1, env.dim)
    cap = eb.default_tree_capacity(md) if capacity is None else capacity
    want = [oracle_api.ray_tree(env, of[i], df[i], (i % w, i // w), md, time, cap) for i in flat]
    assert_trees_equal(got.trees, want, items)
    return got


# ---------------------------------------------------------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", SCENES + ["csg_mix_3d", "no_void_3d"])
def test_trees_equal_oracle(built_lib, name, pipeline, precision):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    env.precision = precision
    check_render_trees(env, (64, 40), time=0.5, seed=sum(name.encode()))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "csg_mix_3d"])
def test_wavefront_equals_megakernel(built_lib, name):
    env = load(name)
    pixels = sample_pixels(48, 30, seed=9)
    runs = []
    for pipeline in ("wavefront", "megakernel"):
        env.pipeline = pipeline_id(pipeline)
        runs.append(env.render((48, 30), 0.25, trees=pixels).trees)
    assert_trees_equal(runs[0], runs[1], pixels)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("depth", [0, 1, 16])
def test_max_depths(built_lib, depth, pipeline):
    env = load("3d_fresnel")
    env.camera.max_depth = depth
    env.pipeline = pipeline_id(pipeline)
    got = check_render_trees(env, (40, 24), seed=depth, capacity=None if depth < 16 else 3000)
    assert max(int(t.nodes["level"].max()) for t in got.trees) <= depth


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["3d_room", "4d_room"])
def test_moved_and_turned_camera(built_lib, name):
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
    check_render_trees(env, (61, 37), time=0.75, seed=4)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_camera_in_no_entity_gives_checkerboard_roots(built_lib, pipeline):
    env = load("no_void_3d")
    env.pipeline = pipeline_id(pipeline)
    got = check_render_trees(env, (37, 23), seed=2)
    for tr in got.trees:
        assert tr.count == 1 and tr.nodes[0]["flags"] == _capi.EUCL_TREE_CHECKERBOARD and tr.nodes[0]["medium"] == -1
        assert np.isnan(tr.nodes[0]["t"]) and np.isnan(tr.nodes[0]["origin"][:3]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_batch_of_traced_and_untraced_frames(built_lib, pipeline):
    env = load("no_void_3d")
    env.pipeline = pipeline_id(pipeline)
    outside = env.camera.copy()  # the scene's camera lies in no entity
    inside = env.camera.copy()
    for k, v in enumerate([10.0, 0.0, 0.5]):  # inside the sphere
        inside.location[k] = v
    cams, times = [inside, outside, inside, outside], [0.0, 0.5, 1.0, 1.5]
    inside2 = inside.copy()
    inside2.location[2] = 0.25
    cams[2] = inside2
    w, h = 40, 24
    items = [(k, x, y) for k in range(4) for x, y in sample_pixels(w, h, seed=k, n=12)]
    plain = env.render_frames((w, h), cams, times, want_hit_ids=True, aovs=ALL)
    got = env.render_frames((w, h), cams, times, want_hit_ids=True, trees=items)
    assert np.array_equal(got.data, plain.data) and np.array_equal(got.hit_ids, plain.hit_ids)
    assert counted(got.stats) == counted(plain.stats)
    check_consistency(env, got.trees, [(k, y, x) for k, x, y in items], plain.data, plain.hit_ids, plain.aovs,
                      int(env.camera.max_depth))
    want = [oracle_api.pixel_trees(env, w, h, [(x, y)], times[k], camera=cams[k], capacity=eb.default_tree_capacity(env.camera.max_depth))[0]
            for k, x, y in items]
    assert_trees_equal(got.trees, want, items)
    kinds = {bool(t.nodes[0]["flags"] & _capi.EUCL_TREE_CHECKERBOARD) for t in got.trees}
    assert kinds == {True, False}


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f64", "f32"])
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "csg_mix_3d"])
def test_random_rays(built_lib, name, pipeline, precision):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    env.precision = precision
    o, d = random_rays(env, 1500, seed=sum(name.encode()))
    items = [int(i) for i in np.random.default_rng(1).choice(len(o), 70, replace=False)]
    check_ray_trees(env, o, d, items, time=0.5)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
@pytest.mark.parametrize("name", ["3d_room", "4d_room", "csg_mix_3d"])
def test_degenerate_rays(built_lib, name, pipeline):
    env = load(name)
    env.pipeline = pipeline_id(pipeline)
    dim = env.dim
    loc = [env.camera.location[k] for k in range(dim)]
    unit = [1.0] + [0.0] * (dim - 1)
    rays = [(loc, [0.0] * dim), (loc, [math.nan] + [0.5] * (dim - 1)), (loc, [math.inf] + [0.0] * (dim - 1)),
            (loc, [-math.inf, 1.0] + [0.0] * (dim - 2)), ([math.nan] * dim, unit), ([math.inf] + loc[1:], unit),
            (loc, [1e-300] * dim), (loc, [1e300] * dim)]
    if name == "csg_mix_3d":  # across the LinearSpace void's boundary
        rays += [([x, 0.0, 0.0], [dx, 0.25, 0.0]) for x in (5.0, 5.5, 6.5, 7.0) for dx in (1.0, -1.0, 0.0)]
    o = np.array([r[0] for r in rays], np.float64)
    d = np.array([r[1] for r in rays], np.float64)
    check_ray_trees(env, o, d, list(range(len(o))))


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_origins_in_no_entity_and_flat_list_against_grid(built_lib, pipeline):
    env = load("no_void_3d")
    env.pipeline = pipeline_id(pipeline)
    o, d = random_rays(env, 48 * 40, seed=3)
    o[: len(o) // 2] = [10.0, 0.0, 0.5]  # half of the origins inside the sphere, the rest in no entity
    rng = np.random.default_rng(8)
    flat_items = [int(i) for i in rng.choice(len(o), 70, replace=False)]
    flat = check_ray_trees(env, o, d, flat_items)
    grid_items = [(i // 48, i % 48) for i in flat_items]
    grid = check_ray_trees(env, o.reshape(40, 48, 3), d.reshape(40, 48, 3), grid_items)
    checker = [bool(t.nodes[0]["flags"] & _capi.EUCL_TREE_CHECKERBOARD) for t in flat.trees]
    assert any(checker) and not all(checker)
    for a, b, c in zip(flat.trees, grid.trees, checker):  # only the checkerboard colour depends on the grid width
        if not c:
            assert oracle_api.first_difference(a, b) is None


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_truncation_keeps_prefixes(built_lib, pipeline):
    env = load("3d_fresnel_2")
    env.pipeline = pipeline_id(pipeline)
    pixels = sample_pixels(48, 30, seed=5)
    full = env.render((48, 30), trees=pixels).trees
    assert max(t.count for t in full) > 7
    for cap in (1, 2, 7):
        got = check_render_trees(env, (48, 30), pixels=pixels, capacity=cap)
        for a, b in zip(got.trees, full):
            assert a.count == b.count and len(a.nodes) == min(cap, b.count) and a.truncated == (b.count > cap)
            assert oracle_api.first_difference(a, eb.RayTree(b.nodes[:cap], b.count, b.dim, b.precision)) is None


@pytest.mark.gpu
@pytest.mark.parametrize("chunk_pixels", [97, 640])
def test_items_in_several_chunks(built_lib, monkeypatch, chunk_pixels):
    env = load("3d_room")
    monkeypatch.setenv("EUCL_CHUNK_PIXELS", str(chunk_pixels))
    check_render_trees(env, (64, 40), seed=6)
    o, d = random_rays(env, 2400, seed=5)
    check_ray_trees(env, o, d, [int(i) for i in np.random.default_rng(2).choice(2400, 60, replace=False)])


@pytest.mark.gpu
@pytest.mark.parametrize("split", [1, 2, 3])
def test_split_pipelines(built_lib, monkeypatch, split):
    env = load("3d_room")
    monkeypatch.setenv("EUCL_SPLIT", str(split))
    w, h = 320, 208  # 66560 pixels: split into `split` pipelines
    pixels = sample_pixels(w, h, seed=split, n=40) + [(x, y) for y in (15, 16, 31, 32, 47, 48) for x in (0, 100)]
    got = check_render_trees(env, (w, h), time=0.5, pixels=pixels)
    assert got.stats["launches"] > 0


@pytest.mark.gpu
def test_forced_arena_retry(built_lib, monkeypatch):
    pixels = sample_pixels(48, 31, seed=7)
    plain = load("3d_fresnel_2").render((48, 31), trees=pixels)
    monkeypatch.setenv("EUCL_ARENA_FACTOR_X10", "11")
    tight = load("3d_fresnel_2")
    got = tight.render((48, 31), trees=pixels, profile=True)
    assert got.stats["retries"] > 0
    assert np.array_equal(got.data, plain.data)
    assert_trees_equal(got.trees, plain.trees, pixels)
    check_render_trees(load("3d_fresnel_2"), (48, 31), pixels=pixels)


@pytest.mark.gpu
@pytest.mark.parametrize("pipeline", ["wavefront", "megakernel"])
def test_duplicate_items(built_lib, pipeline):
    env = load("4d_room")
    env.pipeline = pipeline_id(pipeline)
    pixels = [(5, 7), (20, 11), (5, 7), (0, 0), (20, 11), (5, 7)]
    got = check_render_trees(env, (32, 20), pixels=pixels)
    assert oracle_api.first_difference(got.trees[0], got.trees[2]) is None and oracle_api.first_difference(got.trees[0], got.trees[5]) is None
    o, d = random_rays(env, 500, seed=4)
    check_ray_trees(env, o, d, [3, 499, 3, 3, 17, 499])


@pytest.mark.gpu
def test_graphs_around_tree_calls(built_lib):
    env = load("3d_room")
    w, h = 64, 40
    for _ in range(12):  # the scene settles its ray grouping (no graphs while it measures), then replays
        ref = env.render((w, h), 0.5, want_hit_ids=True)
        if ref.stats["graph_replays"]:
            break
    replays = [env.render((w, h), 0.5, want_hit_ids=True).stats["graph_replays"] for _ in range(2)]
    assert replays[-1] > 0
    pixels = sample_pixels(w, h, seed=1)
    t1 = env.render((w, h), 0.5, want_hit_ids=True, trees=pixels)
    assert t1.stats["graph_replays"] == 0
    after = env.render((w, h), 0.5, want_hit_ids=True)
    assert after.stats["graph_replays"] > 0 and np.array_equal(after.data, ref.data)
    t2 = env.render((w, h), 0.5, want_hit_ids=True, trees=pixels)
    assert t2.stats["graph_replays"] == 0
    for a, b in zip(t1.trees, t2.trees):
        assert a.count == b.count and a.nodes.tobytes() == b.nodes.tobytes()
    assert np.array_equal(t1.data, ref.data) and t1.stats["launches"] > ref.stats["launches"]


@pytest.mark.gpu
def test_invalid_arguments_are_rejected(built_lib):
    env = load("3d_room")
    scene = env._device_scene(0)
    lib = eb.lib()
    w, h = 16, 8
    out = np.full((h, w, 3), 77, np.uint8)
    nodes = np.zeros((4, 8), eb.TREE_NODE_DTYPE)
    counts = np.full(4, 9, np.uint32)
    items = np.array([0, 5, 127, 3], np.uint32)
    frames = (eb.EuclFrame * 2)()
    for k in range(2):
        frames[k].camera = env.camera
    opts = eb.EuclRenderOpts(width=w, height=h)

    def query(**kw):
        fields = dict(items=items.ctypes.data, n_items=4, capacity=8, nodes=nodes.ctypes.data, counts=counts.ctypes.data)
        fields.update(kw)
        return _capi.EuclTreeQuery(**fields)

    def render(q, n_frames=1, o=opts, rgb=out):
        return lib.eucl_render_trees(scene, frames, n_frames, C.byref(o), rgb.ctypes.data if rgb is not None else None, None,
                                     C.byref(q) if q is not None else None, C.byref(eb.EuclStats()))

    bad = [query(n_items=0), query(items=None), query(nodes=None), query(counts=None), query(capacity=0),
           query(n_items=70000), query(capacity=(1 << 24) // 4 + 1), query(items=np.array([0, 1, 128, 2], np.uint32).ctypes.data)]
    for q in bad + [None]:
        assert render(q) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), rgb=None) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), o=eb.EuclRenderOpts(width=w, height=h, band_rows=4, band_world=2)) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), o=eb.EuclRenderOpts(width=w, height=h, compact_rows=1)) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), o=eb.EuclRenderOpts(width=0, height=h)) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), o=eb.EuclRenderOpts(width=w, height=h, pipeline=2)) == EUCL_ERR_INVALID_ARGUMENT
    assert render(query(), n_frames=0) == EUCL_ERR_INVALID_ARGUMENT
    o3 = np.zeros((12, 3))
    d3 = np.ones((12, 3))

    def rays(q, **kw):
        fields = dict(origins=o3.ctypes.data, directions=d3.ctypes.data, n=12, width=1, max_depth=10)
        fields.update(kw)
        r = eb.EuclRays(**fields)
        return lib.eucl_trace_ray_trees(scene, C.byref(r), out.ctypes.data, None, C.byref(q) if q is not None else None,
                                        C.byref(eb.EuclStats()))

    small = np.array([0, 5, 11, 3], np.uint32)
    for q in bad[:-1] + [None, query(items=np.array([0, 12, 1, 2], np.uint32).ctypes.data)]:
        assert rays(q) == EUCL_ERR_INVALID_ARGUMENT
    for kw in [dict(n=0), dict(origins=None), dict(width=5), dict(max_depth=64), dict(pipeline=2)]:
        assert rays(query(items=small.ctypes.data), **kw) == EUCL_ERR_INVALID_ARGUMENT, kw
    assert (out == 77).all() and (counts == 9).all()  # rejected before any device work
    assert render(query(items=np.array([0, 1, 127, 2], np.uint32).ctypes.data)) == EUCL_OK
    assert rays(query(items=small.ctypes.data)) == EUCL_OK and (counts != 9).all()


@pytest.mark.gpu
def test_tool_inspect(built_lib, tmp_path):
    scene = ROOT / "assets" / "scenes" / "3d_room.json"
    w, h = 64, 40
    out = tmp_path / "room.png"
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "eucl_render.py"), str(scene), str(out), "--size", str(w), str(h),
                        "--time", "0.5", "--inspect", "10,7", "--inspect", "center"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "[0] root level 0" in r.stdout
    env = eb.load_reference_scene("3d_room")
    got = env.render((w, h), 0.5, trees=[(10, 7), (w // 2, h // 2)])
    for (x, y), tree in zip([(10, 7), (w // 2, h // 2)], got.trees):
        doc = json.loads((tmp_path / f"room.tree_{x}_{y}.json").read_text())
        assert doc["pixel"] == [x, y] and doc["count"] == tree.count
        back = eucl_render.tree_from_json(doc, env.dim)
        assert oracle_api.first_difference(back, tree) is None


# ---------------------------------------------------------------------------------------------------------------- CPU

def test_tree_structs_match_the_c_layout():
    assert C.sizeof(_capi.EuclTreeNode) == 176 and C.sizeof(_capi.EuclTreeQuery) == 32
    assert eb.TREE_NODE_DTYPE.itemsize == 176
    for name in eb.TREE_NODE_DTYPE.names:
        assert eb.TREE_NODE_DTYPE.fields[name][1] == getattr(_capi.EuclTreeNode, name).offset, name
    assert [getattr(_capi.EuclTreeQuery, n).offset for n in ("items", "n_items", "capacity", "nodes", "counts")] == [0, 8, 12, 16, 24]


def test_new_kernels_are_in_the_library(built_lib):
    import test_kernel_resources as kr

    if not Path(kr.CUOBJDUMP).exists() and not shutil.which("cuobjdump"):
        pytest.skip("cuobjdump (CUDA toolkit) not installed")
    names = list(kr.resource_usage(_capi.LIB_PATH))
    for tag in ("k_tree_export", "k_megakernel_tree", "k_megakernel_rays_tree"):
        for ns in ("_ZN4euclANON", "_ZN8eucl_fANON"):  # the f64 and the f32 build, D = 3 and 4 each
            assert sum(1 for k in names if k.startswith(ns + tag + "I")) == 2, (ns, tag)


def test_python_argument_checks():
    env = eb.load_reference_scene("3d_room")
    for bad in ([(64, 0)], [(0, 40)], [(-1, 0)], []):
        with pytest.raises(ValueError):
            env.render((64, 40), trees=bad)
    with pytest.raises(ValueError):
        env.render((64, 40), trees=[(0, 0)], aovs=["depth"])
    with pytest.raises(ValueError):
        env.render((64, 40), trees=[(0, 0)], tree_capacity=0)
    with pytest.raises(ValueError):
        env.render((64, 40), trees=[(0, 0)] * 70000)
    with pytest.raises(ValueError):
        env.render((64, 40), trees=[(0, 0)] * 5000, tree_capacity=4096)
    cams = [env.camera.copy(), env.camera.copy()]
    for bad in ([(2, 0, 0)], [(0, 64, 0)], [(1, 0, 40)]):
        with pytest.raises(ValueError):
            env.render_frames((64, 40), cams, trees=bad)
    with pytest.raises(ValueError):
        env.render_frames((64, 40), cams, trees=[(0, 0, 0)], aovs=["levels"])
    o = np.zeros((4, 6, 3))
    for bad in ([24], [-1], [(4, 0)], [(0, 6)]):
        with pytest.raises(ValueError):
            env.trace_rays(o, o, trees=bad)
    with pytest.raises(ValueError):
        env.trace_rays(o, o, trees=[0], aovs=["depth"])
    assert eb.default_tree_capacity(0) == 1 and eb.default_tree_capacity(10) == 2047 and eb.default_tree_capacity(16) == 4096


def test_ray_tree_helpers():
    nodes = np.zeros(4, eb.TREE_NODE_DTYPE)
    nodes["parent"] = [-1, 0, 1, 0]
    nodes["level"] = [0, 1, 2, 1]
    nodes["kind"] = [0, 1, 2, 2]
    nodes["hit_entity"] = [3, 2, -1, -1]
    nodes["t"] = [2.0, 0.5, np.inf, np.inf]
    nodes["origin"][:, :3] = [1.0, 2.0, 3.0]
    nodes["direction"][:, :3] = [0.5, 0.0, -1.0]
    tree = eb.RayTree(nodes, 9, 3)
    assert tree.truncated and tree.children(0) == [1, 3] and tree.children(1) == [2] and tree.children(3) == []
    p = tree.locations()
    assert np.array_equal(p[0], [2.0, 2.0, 1.0]) and np.array_equal(p[1], [1.25, 2.0, 2.5]) and np.isnan(p[2:]).all()
    text = tree.format().splitlines()
    assert text[0].startswith("[0] root level 0") and text[2].startswith("    [2] reflected level 2") and "5 more" in text[-1]
    other = eb.RayTree(nodes.copy(), 9, 3)
    assert oracle_api.first_difference(tree, other) is None
    other.nodes["t"][1] = np.nextafter(0.5, 1.0)
    assert oracle_api.first_difference(tree, other).startswith("node 1, level 1, transmitted: t 0x3fe0000000000000 vs 0x3fe0000000000001")
    nan2 = eb.RayTree(nodes.copy(), 9, 3)
    nodes["t"][2] = np.nan
    nan2.nodes["t"][2] = -np.float64(np.nan)
    assert oracle_api.first_difference(eb.RayTree(nodes, 9, 3), nan2) is None
    assert "node count 9 vs 8" in oracle_api.first_difference(tree, eb.RayTree(nodes.copy(), 8, 3))


def test_tool_inspect_option_parsing():
    args = eucl_render.parse_args(["s.json", "o.png", "--inspect", "3,4", "--inspect", "center"])
    assert args.inspect == [(3, 4), "center"]
    assert eucl_render.inspect_pixels(args.inspect, 64, 40) == [(3, 4), (32, 20)]
    for bad in (["--inspect", "3"], ["--inspect", "a,b"], ["--inspect", "1,2,3"]):
        with pytest.raises(SystemExit):
            eucl_render.parse_args(["s.json", "o.png", *bad])
    with pytest.raises(SystemExit):
        eucl_render.parse_args(["s.json", "o_%04d.png", "--frames", "3", "--inspect", "1,1"])
    with pytest.raises(SystemExit):
        eucl_render.parse_args(["s.json", "o.png", "--inspect", "1,1", "--aov", "depth"])
    assert eucl_render.parse_args(["s.json", "o.png", "--inspect", "1,1", "--projection", "equirect"]).inspect == [(1, 1)]


@pytest.mark.parametrize("variant", ["det", "f32"])
@pytest.mark.parametrize("name", SCENES)
def test_oracle_restatement_equals_oracle(name, variant):
    """Every pixel of a small frame: the composited root is oracle_render's pixel, the root hit its hit id, the per-level
    node counts the AOV oracle's segments / levels, and the Tracer's level counts those of oracle_render."""
    env = load(name)
    w, h = (16, 10) if variant == "det" else (8, 6)
    rgb, hit, planes, stats = oracle_api.render_aovs(env, w, h, time=0.5, variant=variant)
    pixels = [(x, y) for y in range(h) for x in range(w)]
    trees = oracle_api.pixel_trees(env, w, h, pixels, 0.5, capacity=1 << 14, variant=variant, level_counts=True)
    md = int(env.camera.max_depth)
    total = np.zeros(md + 1, np.uint64)
    for (x, y), (tree, levels) in zip(pixels, trees):
        assert not tree.truncated
        assert np.array_equal(oracle_api.tree_pixel(tree.nodes[0], variant), rgb[y, x]), (x, y)
        assert tree.nodes[0]["hit_entity"] == hit[y, x], (x, y)
        lv = tree.nodes["level"]
        assert np.array_equal(np.bincount(lv, minlength=md + 1), levels), (x, y)
        assert int((lv < md).sum()) == planes["segments"][y, x] and int(lv.max()) + 1 == planes["levels"][y, x], (x, y)
        for j in range(1, len(tree.nodes)):  # pre-order: every parent comes before its children, one level up
            p = tree.nodes[j]["parent"]
            assert 0 <= p < j and tree.nodes[p]["level"] + 1 == tree.nodes[j]["level"]
        total += levels
    assert [int(v) for v in total] == stats["level_counts"]
