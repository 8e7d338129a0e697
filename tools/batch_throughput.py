#!/usr/bin/env python
"""Frames per second of a camera path rendered one frame per call against the same path as ONE batch
(Environment.render_frames_device), in one process, alternating the two ways.

For each workload (scene, frame size, K): K frames with distinct poses (steps through the universe plus turns) and
distinct times.  Every repeat continues the animation in time, so neither way replays a CUDA graph -- as in a real
camera path.  The two ways run on two Environment objects of the same scene, so that each settles (arena, ray-grouping
tuner) at its own size.  Both ways must produce the same bytes; the run fails otherwise.  One JSON line per workload:

    python tools/batch_throughput.py [--out FILE] [--repeats 7] [--warmup 8]
"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import bench  # noqa: E402
import euclider_b200 as eb  # noqa: E402

SIZES = [(128, 96), (480, 270), (1920, 1080)]  # the reference's default frame (1024x768 / resolution 8), ~1/16 HD, HD
KS = [1, 8, 64]
MAX_K_LARGE = 8  # 1920x1080: K <= 8 (the two output buffers of a workload stay small, the run short)


def gpu_identity() -> dict:
    r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, _, power = r.stdout.strip().partition(",")
    return {"gpu": name.strip() or None, "power_limit": power.strip() or None}


def camera_path(env, k):
    cams = []
    step = [0.0] * env.dim
    step[0], step[1] = 0.02, 0.06
    for i in range(k):
        if i:
            env.move_camera(step, 1.0)
            if env.dim == 3:
                env.rotate_yaw(0.01)
            else:
                env.rotate_plane4(0, 1, 0.01)
        cams.append(env.camera.copy())
    return cams


def times_of(repeat, k, dt=1.0 / 25):
    return [(repeat * k + i) * dt for i in range(k)]


def sequential(env, cams, times, out, size):
    w, h = size
    stats = []
    frame_bytes = w * h * 3
    for k, (cam, t) in enumerate(zip(cams, times)):
        env.camera = cam
        stats.append(env.render_device(out.data_ptr() + k * frame_bytes, size, t))
    return stats


def profile_families(st_list):
    keys = ("ms_raygen", "ms_intersect", "ms_shade", "ms_resolve")
    return {key: round(sum(s[key] for s in st_list), 3) for key in keys}


def run_workload(name, size, k, repeats, warmup):
    import torch

    w, h = size
    env_seq, env_batch = eb.load_reference_scene(name), eb.load_reference_scene(name)
    cams = camera_path(eb.load_reference_scene(name), k)
    out_seq = torch.zeros((k, h, w, 3), dtype=torch.uint8, device="cuda")
    out_batch = torch.zeros_like(out_seq)
    rep = 0
    for _ in range(bench.settle_frames(warmup)):  # both ways settle with their own scene objects
        sequential(env_seq, cams, times_of(rep, k), out_seq, size)
        env_batch.render_frames_device(out_batch.data_ptr(), size, cams, times_of(rep, k))
        rep += 1
    torch.cuda.synchronize()
    if not torch.equal(out_seq, out_batch):
        raise AssertionError(f"{name} {w}x{h} K={k}: batched frames differ from sequential ones")
    t_seq, t_batch = [], []
    seq_stats = batch_stats = None
    for _ in range(repeats):
        times = times_of(rep, k)
        rep += 1
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        seq_stats = sequential(env_seq, cams, times, out_seq, size)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        batch_stats = env_batch.render_frames_device(out_batch.data_ptr(), size, cams, times)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        t_seq.append(t1 - t0)
        t_batch.append(t2 - t1)
        if not torch.equal(out_seq, out_batch):
            raise AssertionError(f"{name} {w}x{h} K={k}: batched frames differ from sequential ones")
    segments = sum(s["segments"] for s in seq_stats)
    if segments != batch_stats["segments"]:
        raise AssertionError(f"{name} {w}x{h} K={k}: segment counts differ")
    # per-stage device times (profile mode: an event after every launch, one pipeline), one call each way
    times = times_of(rep, k)
    prof_seq = []
    for i, (cam, t) in enumerate(zip(cams, times)):
        env_seq.camera = cam
        prof_seq.append(env_seq.render_device(out_seq.data_ptr() + i * w * h * 3, size, t, profile=True))
    prof_batch = env_batch.render_frames_device(out_batch.data_ptr(), size, cams, times, profile=True)

    def rate(ts):
        med = float(np.median(ts))
        return {"fps_median": round(k / med, 2), "fps_min": round(k / max(ts), 2), "fps_max": round(k / min(ts), 2),
                "mrays_per_s": round(segments / med / 1e6, 2), "ms_per_call_median": round(med * 1e3, 3)}

    seq, bat = rate(t_seq), rate(t_batch)
    return {"scene": name, "width": w, "height": h, "frames": k, "repeats": repeats,
            "sequential": {**seq, "calls": k, "launches": sum(s["launches"] for s in seq_stats),
                           "graph_replays": sum(s["graph_replays"] for s in seq_stats),
                           "profile_ms": {**profile_families(prof_seq), "total": round(sum(s["ms_total"] for s in prof_seq), 3)}},
            "batched": {**bat, "calls": 1, "launches": batch_stats["launches"], "graph_replays": batch_stats["graph_replays"],
                        "profile_ms": {**profile_families([prof_batch]), "total": round(prof_batch["ms_total"], 3)}},
            "speedup_median": round(seq["ms_per_call_median"] / bat["ms_per_call_median"], 3),
            "segments_per_batch": segments, "bytes_equal": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON lines to this file")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--scenes", nargs="+", default=["3d_room", "4d_room"])
    args = ap.parse_args()
    if eb.lib().eucl_device_count() < 1:
        raise SystemExit("batch_throughput.py needs a CUDA device")
    ident = gpu_identity()
    lines = []
    for name in args.scenes:
        for size in SIZES:
            for k in KS:
                if size == (1920, 1080) and k > MAX_K_LARGE:
                    continue
                rec = {**run_workload(name, size, k, args.repeats, args.warmup), **ident}
                line = json.dumps(rec)
                print(line, flush=True)
                lines.append(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
