#!/usr/bin/env python
"""Throughput of the universe queries (Environment.locate, Environment.trace_paths) against the one-at-a-time path.

    python tools/query_throughput.py [--out profiles/r3_query_throughput.json] [--reps 7]

Workloads, one JSON line each (the card's name and power limit are read in the same run and written with every line):
  locate       a 4096 x 4096 grid of points (the --section plane through the camera, 60 units wide) in 3d_room and a
               4096 x 4096 slice of 4d_room: Mpoints/s of the host call (arrays in host memory, staged in chunks) and of the
               device call (torch tensors); the two arms' entity maps must be equal
  trace_paths  2^20 random walkers x 1 step of length 20 in 3d_hallways and 4d_room: walkers/s of one trace_paths call,
               against 1000 sequential eucl_trace_path calls scaled up (walkers/s); the first 1000 walkers' results must
               equal the sequential calls' bit for bit
  camera_path  a 64-frame camera path through 3d_hallways (63 steps of --move 0 0.5 0, as tools/eucl_render.py --frames
               64 makes it): one trace_paths call against 63 move_camera calls, ms; the two arms' locations must be equal
Every arm is warmed up first; the arms of a workload alternate within each of the --reps repetitions, and the median,
minimum and maximum over the repetitions are reported.  Timings are host clocks around synchronous calls.
"""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

import euclider_b200 as eb  # noqa: E402
from eucl_render import section_points  # noqa: E402


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, limit = (v.strip() for v in out.split(","))
    return {"gpu": name, "power_limit_w": float(limit)}


def timed(fn) -> float:
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def spread(values, scale=1.0) -> dict:
    v = [x * scale for x in values]
    return {"median": statistics.median(v), "min": min(v), "max": max(v)}


def alternate(arms: dict, reps: int) -> dict:
    """Seconds per call of each arm: every arm once as warm-up, then `reps` rounds in which the arms alternate."""
    for fn in arms.values():
        fn()
    times = {k: [] for k in arms}
    for _ in range(reps):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    return times


def locate_workload(name: str, reps: int, info: dict) -> dict:
    import torch

    env = eb.load_reference_scene(name)
    pts = section_points(env.camera, env.dim, 4096, 4096, 60.0).reshape(-1, env.dim)
    n = len(pts)
    d_pts = torch.from_numpy(pts).cuda()
    d_out = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    res = {}
    times = alternate({"host": lambda: res.__setitem__("host", env.locate(pts)),
                       "device": lambda: env.locate_device(d_pts.data_ptr(), n, d_out.data_ptr())}, reps)
    equal = bool(np.array_equal(res["host"], d_out.cpu().numpy()))
    entities = sorted(int(e) for e in np.unique(res["host"]))
    return {"workload": "locate", "scene": name, "points": n, "unit": "Mpoints/s", "entities": entities,
            "host": spread([n / t / 1e6 for t in times["host"]]), "device": spread([n / t / 1e6 for t in times["device"]]),
            "outputs_equal": equal, **info}


def trace_paths_workload(name: str, reps: int, info: dict, n: int = 1 << 20, sequential: int = 1000) -> dict:
    env = eb.load_reference_scene(name)
    rng = np.random.default_rng(1)
    dim = env.dim
    loc = rng.uniform(-8.0, 28.0, (n, dim))
    loc[:, 2] = rng.uniform(-3.5, 5.0, n)
    d = rng.normal(size=(n, dim))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    res = {}

    def bulk():
        res["bulk"] = env.trace_paths(loc, d, 20.0)

    def one_by_one():
        res["seq"] = [env.trace_path_unknown(loc[i], d[i], 20.0) for i in range(sequential)]

    times = alternate({"trace_paths": bulk, "sequential": one_by_one}, reps)
    bl, bd, bs = res["bulk"]
    equal = True
    for i, r in enumerate(res["seq"]):
        if r is None:
            equal &= bool(bs[i, 0] == 0)
        else:
            equal &= bool(bs[i, 0] == 1 and np.array_equal(bl[i, 0], r[0]) and np.array_equal(bd[i, 0], r[1]))
    return {"workload": "trace_paths", "scene": name, "walkers": n, "steps": 1, "distance": 20.0, "unit": "walkers/s",
            "trace_paths": spread([n / t for t in times["trace_paths"]]),
            "sequential_eucl_trace_path": spread([sequential / t for t in times["sequential"]]),
            "sequential_calls": sequential, "moved": int((bs == 1).sum()), "in_no_entity": int((bs == 0).sum()),
            "outputs_equal": equal, **info}


def camera_path_workload(reps: int, info: dict, frames: int = 64) -> dict:
    env = eb.load_reference_scene("3d_hallways")
    start = env.camera.copy()
    move = [0.0, 0.5, 0.0]
    res = {}

    def one_call():
        unit, dist = eb.camera_step(move, 1.0, env.dim)
        locs, _, _ = env.trace_paths([start.location[k] for k in range(3)], unit, dist, steps=frames - 1)
        res["one"] = locs

    def per_frame():
        env.camera = start.copy()
        locs = []
        for _ in range(frames - 1):
            env.move_camera(move, 1.0)
            locs.append([env.camera.location[k] for k in range(3)])
        res["loop"] = np.array(locs)

    times = alternate({"trace_paths": one_call, "move_camera": per_frame}, reps)
    return {"workload": "camera_path", "scene": "3d_hallways", "frames": frames, "steps": frames - 1, "move": move,
            "unit": "ms", "trace_paths": spread(times["trace_paths"], 1e3), "move_camera": spread(times["move_camera"], 1e3),
            "outputs_equal": bool(np.array_equal(res["one"], res["loop"])), **info}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r3_query_throughput.json"))
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if eb.lib().eucl_device_count() < 1:
        raise SystemExit("query_throughput needs a CUDA device")
    info = gpu_info()
    rows = [locate_workload("3d_room", args.reps, info), locate_workload("4d_room", args.reps, info),
            trace_paths_workload("3d_hallways", args.reps, info), trace_paths_workload("4d_room", args.reps, info),
            camera_path_workload(args.reps, info)]
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    with open(args.out, "w") as f:
        for r in rows:
            line = json.dumps(r)
            print(line)
            f.write(line + "\n")
    if not all(r["outputs_equal"] for r in rows):
        raise SystemExit("the arms of a workload disagree")


if __name__ == "__main__":
    main()
