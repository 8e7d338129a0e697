#!/usr/bin/env python
"""What the per-pixel auxiliary outputs cost: a plain render against the same render with all five AOV planes
(depth, position, normal, segments, levels), both into device buffers, in one process on one Environment per way.

After a warm-up (arena sizing, the ray-grouping tuner, the graph capture) the two ways alternate call by call,
--repeats times each; every call replays its way's CUDA graph, as a repeated benchmark frame does.  Timed is the device
time of each call (EuclStats.ms_total).  The frames of both ways must be equal bytes and the segments plane must sum to
the frame's segment count; the run fails otherwise.  One JSON line per workload:

    python tools/aov_overhead.py [--out FILE] [--repeats 20]
"""
import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import euclider_b200 as eb  # noqa: E402
from batch_throughput import gpu_identity  # noqa: E402

WORKLOADS = [("3d_room", 3840, 2160), ("4d_room", 7680, 4320)]


def measure(name, w, h, repeats):
    import torch

    plain_env, aov_env = eb.load_reference_scene(name), eb.load_reference_scene(name)
    dim = plain_env.dim
    rgb = {way: torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda") for way in ("plain", "aovs")}
    planes = {"depth": torch.empty((h, w), dtype=torch.float32, device="cuda"),
              "position": torch.empty((h, w, dim), dtype=torch.float32, device="cuda"),
              "normal": torch.empty((h, w, dim), dtype=torch.float32, device="cuda"),
              "segments": torch.empty((h, w), dtype=torch.int32, device="cuda"),  # uint32 bytes
              "levels": torch.empty((h, w), dtype=torch.int32, device="cuda")}
    d_aovs = {n: t.data_ptr() for n, t in planes.items()}

    def call(way):
        if way == "plain":
            return plain_env.render_device(rgb[way].data_ptr(), (w, h))
        return aov_env.render_device(rgb[way].data_ptr(), (w, h), d_aovs=d_aovs)

    for _ in range(8):
        for way in ("plain", "aovs"):
            call(way)
    ms = {"plain": [], "aovs": []}
    replays = {"plain": 0, "aovs": 0}
    for _ in range(repeats):
        for way in ("plain", "aovs"):
            st = call(way)
            ms[way].append(st["ms_total"])
            replays[way] += st["graph_replays"]
    if not torch.equal(rgb["plain"], rgb["aovs"]):
        raise SystemExit(f"{name} {w}x{h}: the frame with AOVs differs from the plain frame")
    segments = int(planes["segments"].to(torch.int64).sum().item())
    st = plain_env.render_device(rgb["plain"].data_ptr(), (w, h))
    if segments != st["segments"]:
        raise SystemExit(f"{name}: sum of the segments plane {segments} != stats {st['segments']}")
    med = {way: statistics.median(v) for way, v in ms.items()}
    return {"scene": name, "width": w, "height": h, "timed_calls": len(ms["plain"]),
            "plain_ms_median": round(med["plain"], 4), "aovs_ms_median": round(med["aovs"], 4),
            "plain_ms_min": round(min(ms["plain"]), 4), "aovs_ms_min": round(min(ms["aovs"]), 4),
            "overhead_ms": round(med["aovs"] - med["plain"], 4), "overhead_pct": round(100.0 * (med["aovs"] / med["plain"] - 1.0), 2),
            "graph_replays": replays, "aov_bytes_written": w * h * (12 + 8 * dim)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=20)
    args = ap.parse_args()
    ident = gpu_identity()
    lines = []
    for name, w, h in WORKLOADS:
        rec = {**measure(name, w, h, args.repeats), **ident, "command": " ".join(["python", "tools/aov_overhead.py"] + sys.argv[1:])}
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
