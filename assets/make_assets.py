#!/usr/bin/env python
"""Writes the benchmark and test scenes (assets/scenes/*.json) and their textures (assets/resources/*.png).

The ten scenes are restatements, in the reference's JSON constructor vocabulary, of the scenes that ship with
Limeth/euclider, following the descriptions in SURVEY.md (Appendix B).  The six benchmark scenes have the same
entities in the same order, the same primitive counts, camera poses and materials; the four others (3d_frame,
3d_fresnel_2, 3d_photo, 4d_fresnel) follow the survey's shorter descriptions.  Where the survey leaves a colour or a
detail open, a value is chosen here.

The reference's JPEG textures are not redistributed; the PNG textures written here are procedural stand-ins of the
same role (a UV test grid, a star field, a 32x32 black-and-white pattern).  They are build products: build() in
__graft_entry__.py writes them (`--textures`) into the git-ignored assets/resources/.  Every texel comes from exact
arithmetic and PNG is lossless, so every machine renders the same frames (tests/golden depends on it).

The scenes are committed; run this from the repository root without arguments only to change them, then refresh
tests/golden with tools/make_golden.py:
    python assets/make_assets.py [--textures]
"""
import json
import sys
from pathlib import Path

import numpy as np
from PIL import Image

HERE = Path(__file__).resolve().parent
UV_GRID = "./resources/uv_grid.png"
STARS = "./resources/stars.png"
SIMPLE = "./resources/simple.png"


def P(*c): return {f"Point{len(c)}::new": list(c)}
def V(*c): return {f"Vector{len(c)}::new": list(c)}
def rgba(r, g, b, a): return {"Rgba::new": [r, g, b, a]}
def hsva(h, s, v, a): return {"Rgba::from_hsva": [h, s, v, a]}
def op(name): return {"SetOperation": [name]}
def of(d, shapes, name): return {f"ComposableShape{d}::of": [shapes, op(name)]}
def vac(d): return {f"Vacuum{d}::new": []}
def void(d): return {f"Void{d}::new_with_vacuum": []}
def entity(d, shape, surf, material=None): return {f"Entity{d}Impl::new": [shape, material or vac(d), surf]}
def cuboid(c, dims): return {"HalfSpace3::cuboid": [P(*c), V(*dims)]}
def hypercuboid(c, dims): return {"HalfSpace4::hypercuboid": {"center": P(*c), "dimensions": V(*dims)}}


def halfspace(normal, through, inside):
    d = len(normal)
    return {f"HalfSpace{d}::new_with_point": [{f"Hyperplane{d}::new_with_point": [V(*normal), P(*through)]}, P(*inside)]}


def surface(d, ratio, color, threshold=None):
    return {f"ComposableSurface{d}": {
        "reflection_ratio": ratio, "reflection_direction": {f"reflection_direction_specular_{d}": []},
        "threshold_direction": threshold or {f"threshold_direction_identity_{d}": []}, "surface_color": color}}


def uniform_ratio(d, r): return {f"reflection_ratio_uniform_{d}": [r]}
def uniform(d, c): return {f"surface_color_uniform_{d}": [c]}
def blend(d, src, dst, fn): return {f"surface_color_blend_{d}": [src, dst, {f"blend_function_{fn}": []}]}
def illum_global(d): return {f"surface_color_illumination_global_{d}": [rgba(1, 1, 1, 0), rgba(0, 0, 0, 0.5)]}
def illum_dir(d, direction, light, dark): return {f"surface_color_illumination_directional_{d}": [V(*direction), light, dark]}
def shaded(d, color): return blend(d, illum_global(d), color, "darken")  # global illumination darkening a colour


def glass(d, snell=True):
    """Fresnel(1.458, 1) glass, specular reflection, Snell refraction (or none), no colour of its own."""
    thr = {f"threshold_direction_snell_{d}": [1.458]} if snell else None
    return surface(d, {f"reflection_ratio_fresnel_{d}": [1.458, 1.0]}, uniform(d, rgba(0, 0, 0, 0)), thr)


def background(d, path, filt="texture_image_linear"):
    uv = {"uv_sphere_3": [P(0, 0, 0)]}
    if d == 4:
        uv = {"uv_derank_4": [uv]}
    return {f"MappedTextureImpl{d}::new": [uv, {filt: [path]}]}


def universe(d, camera, entities, bg):
    return {f"Universe{d}": {"camera": camera, "entities": entities + [void(d)], "background": bg}}


def fresnel_3d():
    return universe(3, {"PitchYawCamera3": []}, [entity(3, {"Sphere3::new": [P(10, 0, 0), 3]}, glass(3))],
                    background(3, UV_GRID))


def fresnel_4d():
    return universe(4, {"FreeCamera4": []}, [entity(4, {"Sphere4::new": [P(10, 0, 0, 0), 3]}, glass(4))],
                    background(4, UV_GRID))


def fresnel_2_3d():
    """A glass sphere bored through by a vertical cylinder: the inner walls branch the ray tree at every level."""
    shape = of(3, [{"Sphere3::new": [P(10, 0, 0), 3]}, {"Cylinder3::new": [P(10, 0, 0), V(0, 0, 1), 1]}], "Complement")
    return universe(3, {"PitchYawCamera3": []}, [entity(3, shape, glass(3))], background(3, SIMPLE, "texture_image_nearest_neighbor"))


def room_3d():
    d = 3
    walls = of(d, [halfspace((0, 0, 1), (0, 0, -4), (0, 0, -5)), halfspace((0, 0, 1), (0, 0, 6), (0, 0, 7)),
                   halfspace((1, 0, 0), (19, 0, 0), (20, 0, 0)), halfspace((1, 0, 0), (-1, 0, 0), (-2, 0, 0))], "Union")
    perlin = blend(d, {"surface_color_perlin_hue_random_3": [5, 0.1]}, {"surface_color_perlin_hue_random_3": [2, 0.3]},
                   "difference")
    ents = [
        entity(d, {"Sphere3::new": [P(14, 5, -1), 3]}, surface(d, uniform_ratio(d, 0.5), shaded(d, uniform(d, rgba(0, 0, 1, 0.25))))),
        entity(d, cuboid((16, 0, -1), (3, 3, 6)), surface(d, uniform_ratio(d, 0), shaded(d, perlin))),
        entity(d, {"Cylinder3::new": [P(8, -6, 0), V(1, 1, 4), 1]}, glass(d)),
        entity(d, of(d, [cuboid((14, -6, -2), (4, 4, 4)), {"Sphere3::new": [P(14, -6, -2), 2.5]}], "Complement"), glass(d)),
        entity(d, halfspace((0, 1, 0), (0, -10, 0), (0, -11, 0)), surface(d, uniform_ratio(d, 0), shaded(d, uniform(d, rgba(1, 0, 0, 1))))),
        entity(d, halfspace((0, 1, 0), (0, 10, 0), (0, 11, 0)), surface(d, uniform_ratio(d, 0), shaded(d, uniform(d, rgba(0, 1, 0, 1))))),
        entity(d, walls, surface(d, uniform_ratio(d, 0), shaded(d, illum_dir(d, (0, 0, -1), rgba(1, 1, 1, 1), rgba(0.5, 0.5, 0.5, 1))))),
    ]
    return universe(d, {"PitchYawCamera3": []}, ents, background(d, STARS))


def hallways_3d():
    """Two hallways, each walled by a shell: the left one's void stretches x fourfold, the right one's shrinks it."""
    d = 3

    def space(fwd, inv):
        exprs = [{"ComponentTransformationExpr": [fwd, inv]}, {"ComponentTransformationExpr": ["y", "y"]},
                 {"ComponentTransformationExpr": ["z", "z"]}]
        return {"LinearSpace3": ["xyz", [{"ComponentTransformation3": [exprs]}]]}

    portal = surface(d, uniform_ratio(d, 0), uniform(d, rgba(0, 0, 0, 0)))

    def shell(c, length, color):
        return entity(d, of(d, [cuboid(c, (length, 5, 8)), cuboid(c, (length + 1.01, 3.01, 6.01))], "Complement"),
                      surface(d, uniform_ratio(d, 0), shaded(d, illum_dir(d, (0, 0, -1), color, rgba(0, 0, 0, 1)))))

    ents = [
        entity(d, cuboid((20, -5, -1), (20, 3, 6)), portal, space("x * 4", "x / 4")),
        shell((20, -5, -1), 20, rgba(0.2, 0.4, 1, 1)),
        entity(d, cuboid((20, 5, -1), (5, 3, 6)), portal, space("x / 4", "x * 4")),
        shell((20, 5, -1), 5, rgba(1, 0.6, 0.1, 1)),
        entity(d, halfspace((0, 0, 1), (0, 0, -4), (0, 0, -5)), surface(d, uniform_ratio(d, 0), shaded(d, uniform(d, rgba(0.6, 0.6, 0.6, 1))))),
    ]
    return universe(d, {"PitchYawCamera3": []}, ents, background(d, STARS))


def frame_surface(d):
    light = (0, 0, -1) if d == 3 else (0, 0, -1, 0)
    return surface(d, uniform_ratio(d, 0), shaded(d, illum_dir(d, light, rgba(1, 1, 1, 1), rgba(0.25, 0.25, 0.25, 1))))


def frame_3d():
    """The cube frame: a cube with three crossing square tunnels carved out; the camera sits at the crossing."""
    bars = of(3, [cuboid((0, 0, 0), (5, 3, 3)), cuboid((0, 0, 0), (3, 5, 3)), cuboid((0, 0, 0), (3, 3, 5))], "Union")
    shape = of(3, [cuboid((0, 0, 0), (4, 4, 4)), bars], "Complement")
    return universe(3, {"FreeCamera3": []}, [entity(3, shape, frame_surface(3))], background(3, UV_GRID))


def frame_4d():
    """The hypercube frame: the four-dimensional counterpart of 3d_frame (40 half-spaces)."""
    bars = of(4, [hypercuboid((0, 0, 0, 0), dims) for dims in ((5, 3, 3, 3), (3, 5, 3, 3), (3, 3, 5, 3), (3, 3, 3, 5))], "Union")
    shape = of(4, [hypercuboid((0, 0, 0, 0), (4, 4, 4, 4)), bars], "Complement")
    return universe(4, {"FreeCamera4": []}, [entity(4, shape, frame_surface(4))], background(4, UV_GRID))


def cylinders_4d():
    """The edges of a tesseract of side 4 as capped cylinders, its vertices as spheres: the eight vertices with an
    odd number of negative coordinates form entity 0; each even vertex is one entity with its four edges."""
    d = 4
    corners = [tuple(2 * (1 - 2 * ((k >> i) & 1)) for i in range(4)) for k in range(16)]
    odd = [c for c in corners if sum(v < 0 for v in c) % 2]
    even = [c for c in corners if not sum(v < 0 for v in c) % 2]

    def look(hue):
        return surface(d, uniform_ratio(d, 0.2), shaded(d, illum_dir(d, (0, 0, -1, 0), hsva(hue, 0.8, 1, 1), hsva(hue, 0.8, 0.3, 1))))

    ents = [entity(d, of(d, [{"Sphere4::new": [P(*c), 0.5]} for c in odd], "Union"), look(0))]
    for k, c in enumerate(even):
        parts = [{"Sphere4::new": [P(*c), 0.5]}]
        for axis in range(4):
            mid = list(c)
            mid[axis] = 0
            direction = [0, 0, 0, 0]
            direction[axis] = 1
            parts.append({"Cylinder4::new_with_height": [P(*mid), V(*direction), 0.5, 4]})
        ents.append(entity(d, of(d, parts, "Union"), look(45 * (k + 1))))
    return universe(d, {"FreeCamera4": []}, ents, background(d, UV_GRID))


def room_4d():
    d = 4
    r = 4.24264068712

    def mirror(hue):
        return surface(d, uniform_ratio(d, 0.5), shaded(d, uniform(d, hsva(hue, 0.9, 1, 0.5))))

    def opaque(hue):
        return surface(d, uniform_ratio(d, 0), shaded(d, uniform(d, hsva(hue, 0.6, 0.9, 1))))

    box = hypercuboid((0, 0, 0, 0), (40, 40, 20, 20))
    walls = of(d, [{"VoidShape4": []}, box], "Complement")
    ents = [
        entity(d, {"Sphere4::new": [P(15, 0, 0, 0), 3]}, mirror(0)),
        entity(d, {"Sphere4::new": [P(15, 0, r, r), 3]}, mirror(120)),
        entity(d, {"Sphere4::new": [P(15, 6, 0, 0), 3]}, mirror(240)),
        entity(d, hypercuboid((10, -10, -5, 5), (6, 6, 6, 6)), glass(d, snell=False)),
        entity(d, hypercuboid((-10, 10, -5, 5), (8, 8, 8, 8)), opaque(60)),
        entity(d, {"Cylinder4::new": [P(0, 0, 0, 0), V(1, 1, 1, 1), 2]}, opaque(180)),
        entity(d, walls, surface(d, uniform_ratio(d, 0), shaded(d, illum_dir(d, (0, 0, -1, 0), rgba(1, 1, 1, 1), rgba(0.3, 0.3, 0.3, 1))))),
    ]
    return universe(d, {"FreeCamera4::new_with_location": [P(-10, 0, 0, 0)]}, ents, background(d, UV_GRID))


def photo_3d():
    """A glass puck (a vertical cylinder cut by three half-spaces) in front of the camera, a mirror slab behind it."""
    d = 3
    puck = of(d, [{"Cylinder3::new": [P(10, 0, 0), V(0, 0, 1), 3]}, halfspace((0, 0, 1), (0, 0, 2), (0, 0, 1)),
                  halfspace((0, 0, 1), (0, 0, -2), (0, 0, -1)), halfspace((1, 0, 1), (11, 0, 0), (10, 0, 0))], "Intersection")
    ents = [
        entity(d, cuboid((-6, 0, 0), (2, 8, 8)), surface(d, uniform_ratio(d, 0.5), shaded(d, uniform(d, rgba(0.8, 0.8, 0.8, 1))))),
        entity(d, puck, glass(d)),
    ]
    return universe(d, {"PitchYawCamera3": []}, ents, background(d, UV_GRID))


SCENES = {"3d_fresnel": fresnel_3d, "3d_fresnel_2": fresnel_2_3d, "3d_room": room_3d, "3d_hallways": hallways_3d,
          "3d_frame": frame_3d, "3d_photo": photo_3d, "4d_frame": frame_4d, "4d_cylinders": cylinders_4d,
          "4d_room": room_4d, "4d_fresnel": fresnel_4d}


def uv_grid_png(path, size=512):
    """A UV test grid: 16 x 16 cells, hue along u, brightness along v, dark lines between cells (integers only)."""
    yy, xx = np.mgrid[0:size, 0:size]
    cell = size // 16
    cu, cv = xx // cell, yy // cell
    # hsv -> rgb at full saturation, hue = cu / 16 of the circle, in sixteenths of a sextant
    k = (cu * 6)[..., None] + np.array([0, 64, 32])
    t = np.clip(np.minimum(k % 96, 64 - k % 96), 0, 16)
    rgb = (16 - t) * 255 // 16 * (525 + 65 * cv[..., None]) // 1500  # brightness 0.35 .. 1 along v
    rgb[(xx % cell < 2) | (yy % cell < 2)] = 25
    Image.fromarray(rgb.astype(np.uint8), "RGB").save(path, optimize=True)


def stars_png(path, width=1024, height=512, n_stars=3000):
    """A star field: a dark blue sky brightening towards the bottom, and stars whose position, brightness and tint
    come from a 32-bit linear congruential generator (integer arithmetic only, the same on every machine)."""
    blue = 5 + 25 * np.arange(height, dtype=np.int64) // (height - 1)
    img = np.zeros((height, width, 3), np.int64)
    img[...] = np.stack([blue * 2 // 5, blue // 2, blue], axis=-1)[:, None, :]
    state = 2024

    def draw(n):
        nonlocal state
        state = (state * 1664525 + 1013904223) % 2**32
        return (state >> 8) % n

    for _ in range(n_stars):
        y, x, brightness = draw(height), draw(width), 102 + draw(154)
        img[y, x] = [brightness * (204 + draw(52)) // 255 for _ in range(3)]
    Image.fromarray(img.astype(np.uint8), "RGB").save(path, optimize=True)


def simple_png(path):
    """32 x 32 greyscale, only 0 and 255: a checkerboard of 4-pixel squares with a white border."""
    y, x = np.mgrid[0:32, 0:32]
    img = (((x // 4) + (y // 4)) % 2 * 255).astype(np.uint8)
    img[[0, -1], :] = img[:, [0, -1]] = 255
    Image.fromarray(img, "L").save(path, optimize=True)


def write_textures():
    (HERE / "resources").mkdir(exist_ok=True)
    uv_grid_png(HERE / UV_GRID)
    stars_png(HERE / STARS)
    simple_png(HERE / SIMPLE)


def main():
    write_textures()
    if "--textures" in sys.argv[1:]:
        return
    (HERE / "scenes").mkdir(exist_ok=True)
    for name, make in SCENES.items():
        (HERE / "scenes" / f"{name}.json").write_text(json.dumps(make(), indent=1) + "\n")


if __name__ == "__main__":
    main()
