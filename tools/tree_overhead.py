#!/usr/bin/env python
"""What a ray-tree call costs: a plain render against the same render that also returns the ray trees of 1, 256 and 4096
pixels at the default capacity (default_tree_capacity(max_depth) nodes each), both with host outputs, in one process on
one Environment per way.

After a warm-up (arena sizing, the ray-grouping tuner, the plain way's graph capture) the ways alternate call by call,
--repeats times each.  The plain calls replay their CUDA graph; tree calls are never captured.  Timed are the host wall
time of each synchronous call (it includes copying the nodes out) and the device time of the call (EuclStats.ms_total).
Every tree call's frame must equal the plain frame bytes; the run fails otherwise.  One JSON line per item count:

    python tools/tree_overhead.py [--out FILE] [--repeats 10]
"""
import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import euclider_b200 as eb  # noqa: E402
from batch_throughput import gpu_identity  # noqa: E402

SCENE, WIDTH, HEIGHT = "3d_room", 1920, 1080
ITEM_COUNTS = (1, 256, 4096)


def measure(repeats):
    envs = {"plain": eb.load_reference_scene(SCENE), "trees": eb.load_reference_scene(SCENE)}
    rng = np.random.default_rng(0)
    items = {n: [(int(x), int(y)) for x, y in zip(rng.integers(0, WIDTH, n), rng.integers(0, HEIGHT, n))] for n in ITEM_COUNTS}
    out = {way: np.zeros((HEIGHT, WIDTH, 3), np.uint8) for way in envs}

    def call(way, n=None):
        t0 = time.perf_counter()
        img = envs[way].render((WIDTH, HEIGHT), out=out[way], trees=items[n] if way == "trees" else None)
        return (time.perf_counter() - t0) * 1e3, img

    for _ in range(8):
        call("plain")
        call("trees", ITEM_COUNTS[0])
    recs = []
    for n in ITEM_COUNTS:
        wall = {"plain": [], "trees": []}
        dev = {"plain": [], "trees": []}
        replays = {"plain": 0, "trees": 0}
        nodes = 0
        for _ in range(repeats):
            for way in ("plain", "trees"):
                ms, img = call(way, n)
                wall[way].append(ms)
                dev[way].append(img.stats["ms_total"])
                replays[way] += img.stats["graph_replays"]
                if way == "trees":
                    nodes = sum(min(t.count, len(t.nodes)) for t in img.trees)
                    if not np.array_equal(out["trees"], out["plain"]):
                        raise SystemExit(f"{n} items: the frame of the tree call differs from the plain frame")
        med = {k: {way: statistics.median(v) for way, v in d.items()} for k, d in (("wall", wall), ("device", dev))}
        cap = eb.default_tree_capacity(envs["trees"].camera.max_depth)
        recs.append({"scene": SCENE, "width": WIDTH, "height": HEIGHT, "items": n, "capacity": cap, "timed_calls": repeats,
                     "plain_wall_ms_median": round(med["wall"]["plain"], 3), "trees_wall_ms_median": round(med["wall"]["trees"], 3),
                     "plain_device_ms_median": round(med["device"]["plain"], 3),
                     "trees_device_ms_median": round(med["device"]["trees"], 3),
                     "wall_overhead_ms": round(med["wall"]["trees"] - med["wall"]["plain"], 3),
                     "device_overhead_ms": round(med["device"]["trees"] - med["device"]["plain"], 3),
                     "nodes_returned": nodes, "node_bytes_copied": n * cap * 176, "graph_replays": replays})
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=10)
    args = ap.parse_args()
    ident = gpu_identity()
    lines = []
    for rec in measure(args.repeats):
        rec = {**rec, **ident, "command": " ".join(["python", "tools/tree_overhead.py"] + sys.argv[1:])}
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
