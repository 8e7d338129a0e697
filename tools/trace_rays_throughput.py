#!/usr/bin/env python
"""What tracing caller-supplied rays costs against rendering the same rays from the camera: render_device of a frame
against trace_rays_device of that frame's own camera rays (width = frame width), plus an equirect panorama of the same
size, all into device buffers, in one process on one Environment per way.

The camera rays come from the CPU oracle's Tracer::ray_vector (tests/oracle_rays.cc), which equals the device's camera
arithmetic bit for bit, so the frame and the traced rays must be equal bytes; the run fails otherwise.  After a warm-up
(arena sizing, the ray-grouping tuner, graph capture) the three ways alternate call by call, --repeats times each; every
call replays its way's CUDA graph.  Timed is the device time of each call (EuclStats.ms_total, CUDA events on the scene's
stream).  One JSON line per workload:

    python tools/trace_rays_throughput.py [--out FILE] [--repeats 7]
"""
import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))
sys.path.insert(0, str(ROOT / "tests"))

import euclider_b200 as eb  # noqa: E402
import oracle_rays_api  # noqa: E402
from batch_throughput import gpu_identity  # noqa: E402

WORKLOADS = [("3d_room", 1920, 1080), ("4d_room", 1920, 1080)]
DEPTH = 10


def measure(name, w, h, repeats):
    import torch

    envs = {way: eb.load_reference_scene(name) for way in ("render", "rays", "equirect")}
    for env in envs.values():
        env.camera.max_depth = DEPTH
    cam_o, cam_d = oracle_rays_api.camera_rays(envs["rays"], w, h)
    eq_o, eq_d = eb.equirect_rays(envs["equirect"].camera, w, h)
    rays = {"rays": (torch.from_numpy(cam_o).cuda(), torch.from_numpy(cam_d).cuda()),
            "equirect": (torch.from_numpy(eq_o).cuda(), torch.from_numpy(eq_d).cuda())}
    rgb = {way: torch.zeros((h, w, 3), dtype=torch.uint8, device="cuda") for way in envs}

    def call(way):
        if way == "render":
            return envs[way].render_device(rgb[way].data_ptr(), (w, h))
        o, d = rays[way]
        return envs[way].trace_rays_device(o.data_ptr(), d.data_ptr(), w * h, rgb[way].data_ptr(), width=w)

    for _ in range(8):
        for way in envs:
            call(way)
    ms = {way: [] for way in envs}
    replays = {way: 0 for way in envs}
    segments = {}
    for _ in range(repeats):
        for way in envs:
            st = call(way)
            ms[way].append(st["ms_total"])
            replays[way] += st["graph_replays"]
            segments[way] = st["segments"]
    if not torch.equal(rgb["render"], rgb["rays"]):
        raise SystemExit(f"{name} {w}x{h}: the traced camera rays differ from the rendered frame")
    if segments["render"] != segments["rays"]:
        raise SystemExit(f"{name}: segment counts differ ({segments['render']} vs {segments['rays']})")
    med = {way: statistics.median(v) for way, v in ms.items()}
    return {"scene": name, "width": w, "height": h, "max_depth": DEPTH, "timed_calls": repeats,
            "render_ms_median": round(med["render"], 4), "rays_ms_median": round(med["rays"], 4),
            "equirect_ms_median": round(med["equirect"], 4),
            "render_ms_min": round(min(ms["render"]), 4), "rays_ms_min": round(min(ms["rays"]), 4),
            "equirect_ms_min": round(min(ms["equirect"]), 4),
            "rays_overhead_pct": round(100.0 * (med["rays"] / med["render"] - 1.0), 2),
            "frame_bytes_equal": True, "segments": segments, "graph_replays": replays,
            "ray_bytes_read": w * h * 2 * envs["rays"].dim * 8}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also append the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=7)
    args = ap.parse_args()
    ident = gpu_identity()
    lines = []
    for name, w, h in WORKLOADS:
        rec = {**measure(name, w, h, args.repeats), **ident,
               "command": " ".join(["python", "tools/trace_rays_throughput.py"] + sys.argv[1:])}
        print(json.dumps(rec), flush=True)
        lines.append(json.dumps(rec))
    if args.out:
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
