#!/usr/bin/env python
"""Headless renderer: scene JSON -> image file (the reference only renders into a window).

    python tools/eucl_render.py assets/scenes/3d_room.json out.png --size 1920 1080 [--time 1.5]
        [--resource-root assets] [--location x y z [w]] [--max-depth N] [--pipeline megakernel]
"""
import argparse
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import euclider_b200 as eb  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("scene")
    ap.add_argument("output")
    ap.add_argument("--size", type=int, nargs=2, default=(1920, 1080))
    ap.add_argument("--time", type=float, default=0.0)
    ap.add_argument("--resource-root", default=str(eb.ASSET_ROOT))
    ap.add_argument("--location", type=float, nargs="+")
    ap.add_argument("--max-depth", type=int)
    ap.add_argument("--resolution", type=int, default=1, help="the reference's resolution divisor")
    ap.add_argument("--pipeline", default="wavefront", choices=["wavefront", "megakernel"])
    args = ap.parse_args()
    env = eb.Parser.default(resource_root=args.resource_root).parse_file(args.scene)
    if args.location:
        for k, v in enumerate(args.location[:env.dim]):
            env.camera.location[k] = v
    if args.max_depth is not None:
        env.camera.max_depth = args.max_depth
    env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL if args.pipeline == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT
    img = env.render(tuple(args.size), args.time, context=eb.SimulationContext(resolution=args.resolution))
    img.save(args.output)
    st = img.stats
    print(f"{args.output}: {img.width}x{img.height}, {st['segments']} ray segments, {st['ms_total']:.2f} ms on the device")


if __name__ == "__main__":
    main()
