#!/usr/bin/env python
"""Headless renderer: scene JSON -> image file (the reference only renders into a window).

    python tools/eucl_render.py assets/scenes/3d_room.json out.png --size 1920 1080 [--time 1.5]
        [--resource-root assets] [--location x y z [w]] [--max-depth N] [--pipeline megakernel]

Image sequences -- a camera path, a turntable, a Perlin animation -- with --frames N: frame k is the pose after k steps
of the per-frame motion and the time --time + k * --time-step; the output name takes a printf pattern.  Frames are
rendered --batch at a time (default: all in one call, Environment.render_frames).

    python tools/eucl_render.py assets/scenes/3d_room.json out_%04d.ppm --size 128 96 --frames 64 \\
        --move 0 0.05 0 --yaw 0.02 --time-step 0.04

Per-pixel auxiliary outputs with --aov depth,position,normal,segments,levels: next to each image `out.png` the tool writes
`out.<plane>.npy` (the plane as the library returns it, row 0 = bottom) and, for the scalar planes, a greyscale preview
`out.<plane>.png` (top-down; depth and levels linear, segments on a log scale; pixels without a value black).

A 360 x 180 degree panorama of the camera's position with --projection equirect (Environment.trace_rays of
euclider_b200.equirect_rays; the centre column looks forward).  The default, perspective, is the camera's own projection.

    python tools/eucl_render.py assets/scenes/3d_room.json pano.png --size 2048 1024 --projection equirect

The ray tree behind chosen pixels with --inspect X,Y (repeatable; `center` is the pixel (width / 2, height / 2), the
reference's debug pixel): every Universe::trace call of the pixel, printed as an indented tree and written to
`out.tree_X_Y.json` (the nodes of EuclTreeNode, include/euclider_b200.h; pixel (X, Y) with row 0 at the bottom).  Single
frames only, perspective or equirect, and not together with --aov.

    python tools/eucl_render.py assets/scenes/3d_room.json out.png --size 640 360 --inspect center --inspect 100,40
"""
import argparse
import json
import os
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import euclider_b200 as eb  # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("scene")
    ap.add_argument("output", help="image path; with --frames > 1 a printf pattern such as out_%%04d.ppm")
    ap.add_argument("--size", type=int, nargs=2, default=(1920, 1080))
    ap.add_argument("--time", type=float, default=0.0)
    ap.add_argument("--resource-root", default=str(eb.ASSET_ROOT))
    ap.add_argument("--location", type=float, nargs="+")
    ap.add_argument("--max-depth", type=int)
    ap.add_argument("--resolution", type=int, default=1, help="the reference's resolution divisor")
    ap.add_argument("--pipeline", default="wavefront", choices=["wavefront", "megakernel"])
    ap.add_argument("--projection", default="perspective", choices=["perspective", "equirect"],
                    help="equirect: a 360 x 180 degree panorama from the camera's position (single frames only)")
    seq = ap.add_argument_group("image sequences (per-frame motion; angles in radians)")
    seq.add_argument("--frames", type=int, default=1, help="frames to render")
    seq.add_argument("--batch", type=int, help="frames per render call (default: all)")
    seq.add_argument("--move", type=float, nargs="+", metavar="D",
                     help="dx dy dz [dw]: camera step per frame through the universe (Environment.move_camera)")
    seq.add_argument("--yaw", type=float, default=0.0, help="3-D: yaw per frame")
    seq.add_argument("--pitch", type=float, default=0.0, help="3-D: pitch per frame")
    seq.add_argument("--roll", type=float, default=0.0, help="3-D: roll per frame")
    seq.add_argument("--plane4", type=float, nargs=3, metavar=("A", "B", "ANGLE"),
                     help="4-D: rotation per frame in the plane of camera axes A and B (0 forward, 1 left, 2 up, 3 ana)")
    seq.add_argument("--time-step", type=float, default=0.0, help="seconds added to the time per frame")
    ap.add_argument("--aov", type=aov_list, default=[], metavar="P,Q,..",
                    help=f"also write these per-pixel planes, from {','.join(eb.AOV_NAMES)}")
    ap.add_argument("--inspect", type=inspect_spec, action="append", default=[], metavar="X,Y|center",
                    help="print the ray tree of this pixel and write it to out.tree_X_Y.json (repeatable)")
    args = ap.parse_args(argv)
    if args.frames < 1:
        ap.error("--frames must be at least 1")
    if args.batch is not None and args.batch < 1:
        ap.error("--batch must be at least 1")
    if args.move is not None and len(args.move) not in (3, 4):
        ap.error("--move takes 3 or 4 components")
    if args.plane4 is not None and (args.plane4[0] != int(args.plane4[0]) or args.plane4[1] != int(args.plane4[1])):
        ap.error("--plane4: A and B are axis indices")
    if args.frames > 1 and "%" not in args.output:
        ap.error("--frames > 1 needs an output pattern such as out_%04d.ppm")
    if args.projection != "perspective" and is_sequence(args):
        ap.error("--projection equirect renders single frames only")
    if args.inspect and is_sequence(args):
        ap.error("--inspect works on single frames only")
    if args.inspect and args.aov:
        ap.error("--inspect and --aov cannot be used together")
    return args


def inspect_spec(text: str):
    """`center` or `X,Y` (integers)."""
    if text == "center":
        return text
    try:
        x, y = (int(v) for v in text.split(","))
    except ValueError:
        raise argparse.ArgumentTypeError(f"--inspect takes X,Y or center, not {text!r}") from None
    return (x, y)


def inspect_pixels(specs, width: int, height: int) -> list:
    return [(width // 2, height // 2) if s == "center" else s for s in specs]


def tree_to_json(tree: "eb.RayTree", pixel) -> dict:
    fields = eb.TREE_NODE_DTYPE.names
    nodes = [{f: (nd[f][:tree.dim].tolist() if nd[f].ndim else nd[f].item()) if f in ("origin", "direction", "normal")
              else (nd[f].tolist() if nd[f].ndim else nd[f].item()) for f in fields} for nd in tree.nodes]
    return {"pixel": list(pixel), "count": tree.count, "truncated": tree.truncated, "precision": tree.precision, "nodes": nodes}


def tree_from_json(doc: dict, dim: int) -> "eb.RayTree":
    nodes = np.zeros(len(doc["nodes"]), eb.TREE_NODE_DTYPE)
    for j, nd in enumerate(doc["nodes"]):
        for f, v in nd.items():
            if f in ("origin", "direction", "normal"):
                nodes[j][f][:dim] = v
            else:
                nodes[j][f] = v
    return eb.RayTree(nodes, int(doc["count"]), dim, doc.get("precision", "f64"))


def write_trees(image_path: str, pixels, trees) -> None:
    for (x, y), tree in zip(pixels, trees):
        print(f"pixel ({x}, {y}): {tree.count} nodes")
        print(tree.format())
        with open(aov_path(image_path, f"tree_{x}_{y}", ".json"), "w") as f:
            json.dump(tree_to_json(tree, (x, y)), f, indent=1)


def aov_list(text: str) -> list:
    names = text.split(",")
    bad = [n for n in names if n not in eb.AOV_NAMES]
    if bad:
        raise argparse.ArgumentTypeError(f"unknown plane(s) {bad}: choose from {','.join(eb.AOV_NAMES)}")
    return names


def aov_path(image_path: str, name: str, ext: str) -> str:
    """out.png -> out.<name><ext>"""
    return f"{os.path.splitext(image_path)[0]}.{name}{ext}"


def preview(name: str, plane: np.ndarray) -> np.ndarray:
    """Greyscale u8 image of a scalar plane, top-down: linear in depth and levels, log in segments; no value -> black."""
    v = plane.astype(np.float64)
    if name == "segments":
        v = np.log1p(v)
    ok = np.isfinite(v)
    lo, hi = (v[ok].min(), v[ok].max()) if ok.any() else (0.0, 0.0)
    scaled = np.where(ok, (v - lo) / (hi - lo) if hi > lo else 1.0, 0.0)
    return np.round(scaled * 255.0).astype(np.uint8)[::-1]


def write_aovs(image_path: str, aovs: dict) -> None:
    from PIL import Image

    for name, plane in aovs.items():
        np.save(aov_path(image_path, name, ".npy"), plane)
        if plane.ndim == 2:
            Image.fromarray(preview(name, plane)).save(aov_path(image_path, name, ".png"))


def is_sequence(args) -> bool:
    """True when the new per-frame options are in use; otherwise the tool renders one frame with Environment.render."""
    return (args.frames > 1 or args.batch is not None or args.move is not None or args.yaw or args.pitch or args.roll
            or args.plane4 is not None or args.time_step or "%" in args.output)


def step_camera(env, args) -> None:
    """One frame's motion: the translation through the universe, then the turns."""
    if args.move is not None and not env.move_camera(args.move, 1.0):
        print("warning: the camera is in no entity; it stays where it is", file=sys.stderr)
    if args.yaw:
        env.rotate_yaw(args.yaw)
    if args.pitch:
        env.rotate_pitch(args.pitch)
    if args.roll:
        env.rotate_roll(args.roll)
    if args.plane4 is not None:
        env.rotate_plane4(int(args.plane4[0]), int(args.plane4[1]), args.plane4[2])


def main(argv=None):
    args = parse_args(argv)
    env = eb.Parser.default(resource_root=args.resource_root).parse_file(args.scene)
    if args.location:
        for k, v in enumerate(args.location[:env.dim]):
            env.camera.location[k] = v
    if args.max_depth is not None:
        env.camera.max_depth = args.max_depth
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL if args.pipeline == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT
    context = eb.SimulationContext(resolution=args.resolution)
    if args.projection == "equirect":
        w, h = args.size[0] // args.resolution, args.size[1] // args.resolution
        pixels = inspect_pixels(args.inspect, w, h)
        res = env.trace_rays(*eb.equirect_rays(env.camera, w, h), args.time, want_hit_ids=False, aovs=args.aov or None,
                             trees=[(y, x) for x, y in pixels] if pixels else None)
        eb.RawImage2d(res.data, w, h).save(args.output)
        if args.aov:
            write_aovs(args.output, res.aovs)
        if pixels:
            write_trees(args.output, pixels, res.trees)
        st = res.stats
        print(f"{args.output}: {w}x{h} equirect, {st['segments']} ray segments, {st['ms_total']:.2f} ms on the device")
        return
    if not is_sequence(args):
        pixels = inspect_pixels(args.inspect, args.size[0] // args.resolution, args.size[1] // args.resolution)
        img = env.render(tuple(args.size), args.time, context=context, aovs=args.aov or None, trees=pixels or None)
        img.save(args.output)
        if args.aov:
            write_aovs(args.output, img.aovs)
        if pixels:
            write_trees(args.output, pixels, img.trees)
        st = img.stats
        print(f"{args.output}: {img.width}x{img.height}, {st['segments']} ray segments, {st['ms_total']:.2f} ms on the device")
        return
    cameras, times = [], []
    for k in range(args.frames):
        if k > 0:
            step_camera(env, args)
        cameras.append(env.camera.copy())
        times.append(args.time + k * args.time_step)
    batch = args.batch or args.frames
    segments, ms = 0, 0.0
    for k0 in range(0, args.frames, batch):
        frames = env.render_frames(tuple(args.size), cameras[k0:k0 + batch], times[k0:k0 + batch], context=context,
                                   aovs=args.aov or None)
        for j in range(len(frames)):
            frames.frame(j).save(args.output % (k0 + j))
            if args.aov:
                write_aovs(args.output % (k0 + j), frames.frame(j).aovs)
        segments += frames.stats["segments"]
        ms += frames.stats["ms_total"]
    print(f"{args.output}: {args.frames} frames of {frames.width}x{frames.height} in calls of {batch}, {segments} ray segments, "
          f"{ms:.2f} ms on the device")


if __name__ == "__main__":
    main()
