#!/usr/bin/env python
"""Headline benchmark: Mrays/s (ray segments per second) and frame time on a reference scene.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scene 3d_room]
                    [--width 3840 --height 2160] [--pipeline wavefront|megakernel] [--no-configs] [--dump-outputs DIR]

A "step" is one fixed-pose headless frame (Environment::render, src/universe/mod.rs:300-357).
 * value    : whole-job ray segments / second with the frame left in HBM (eucl_render_device)
 * e2e      : the same through the reference-facing call with a HOST output buffer
              (Environment.render -> eucl_render; frame copied device->host every step).  At N > 1 every
              rank writes its own row bands into ONE shared pinned host frame over its own PCIe link.
 * roofline : FP64 issue roofline of k_intersect (SURVEY.md section 8(d)), the same definition at every N:
              sum over ranks of segments x F_scene / slowest rank's k_intersect time, against N x the peak
              measured live by a DADD/DMUL/DFMA microbenchmark
 * cpu_baseline : the CPU oracle (restatement of the reference, oracle/) on a bounded sample
 * configs  : every BASELINE.json config measured in the same run (N = 1: all six; N > 1: the headline and
              4d_room 7680x4320 at max_depth 10 and 16)
`--impl reference` times the CPU oracle alone with all host threads, WHOLE frames (the Rust reference
cannot be built here: no rustc/cargo; see DESIGN.md).
N > 1: one process per GPU (torchrun); interleaved row bands, one gather to rank 0, no other
collective -- the frame is fixed, so scaling is "strong".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

# algorithmic lower-bound flops per ray segment (SURVEY.md 8(d)): every primitive of every surfaced
# entity is tested once per segment; Sphere 7D+4, (half)plane 4D, Cylinder 15D+2
PRIM_FLOPS = {1: lambda d: 7 * d + 4, 2: lambda d: 4 * d, 3: lambda d: 4 * d, 4: lambda d: 15 * d + 2}

DEFAULT_CONFIGS = {
    "3d_fresnel": (1920, 1080), "3d_room": (3840, 2160), "3d_hallways": (3840, 2160), "4d_frame": (3840, 2160),
    "4d_cylinders": (3840, 2160), "4d_room": (7680, 4320),
}
# BASELINE.json `configs`, in its order: (scene, width, height, max_depth or 0 = the reference's literal 10)
ALL_CONFIGS = [("3d_fresnel", 1920, 1080, 0, "f64"), ("3d_room", 3840, 2160, 0, "f64"), ("3d_hallways", 3840, 2160, 0, "f64"),
               ("4d_frame", 3840, 2160, 0, "f64"), ("4d_cylinders", 3840, 2160, 0, "f64"), ("4d_room", 7680, 4320, 0, "f64"),
               ("4d_room", 7680, 4320, 16, "f64"),
               # secondary lines: the reference's `low_precision` feature (type F = f32); the headline stays f64
               ("3d_room", 3840, 2160, 0, "f32"), ("4d_room", 7680, 4320, 0, "f32")]
MULTI_GPU_CONFIGS = [("4d_room", 7680, 4320, 0, "f64"), ("4d_room", 7680, 4320, 16, "f64")]


def scene_flops_per_segment(env) -> int:
    flat = env.flat
    total = 0
    for e in range(flat.n_entities):
        ent = flat.entities[e]
        if ent.surface < 0:
            continue
        for n in range(ent.node_first, ent.node_root + 1):
            node = flat.nodes[n]
            if node.op == 0:
                kind = flat.prims[node.prim].kind
                if kind in PRIM_FLOPS:
                    total += PRIM_FLOPS[kind](flat.dim)
    return total


class ClockSampler:
    """Samples SM clocks and throttle reasons with nvidia-smi while the timed region runs."""

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_sample(env, width, height, t, n_blocks=9, rows_per_block=8, threads=None):
    """Times the CPU oracle on `n_blocks` row blocks spread over the frame.
    Returns (segments, seconds, rows actually rendered, description, threads)."""
    import oracle_api

    threads = threads or os.cpu_count() or 1
    rows_per_block = max(1, min(rows_per_block, height))
    n_blocks = max(1, min(n_blocks, height // rows_per_block))
    starts = [int((k + 0.5) * height / n_blocks - rows_per_block / 2) for k in range(n_blocks)]
    segs, secs = 0, 0.0
    for r0 in starts:
        r0 = max(0, min(height - rows_per_block, r0))
        t0 = time.perf_counter()
        _, _, st = oracle_api.render(env, width, height, time=t, threads=threads, rows=(r0, r0 + rows_per_block))
        secs += time.perf_counter() - t0
        segs += st["segments"]
    rows = n_blocks * rows_per_block
    return segs, secs, rows, f"{n_blocks} blocks x {rows_per_block} rows of the {width}x{height} frame, spread evenly", threads


def run_reference(args, width, height):
    """--impl reference: the CPU restatement of the reference's path, all host threads, whole frames
    (`--ref-rows R` > 0 bounds a step to 9 blocks of R rows and extrapolates; the default renders every row)."""
    import euclider_b200 as eb
    import oracle_api

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    env = eb.load_reference_scene(args.scene)
    if args.max_depth:
        env.camera.max_depth = args.max_depth
    threads = os.cpu_count() or 1
    whole = args.ref_rows <= 0
    seg_total, sec_total, rows_total, desc = 0, 0.0, 0, ""

    def one_step():
        if whole:
            t0 = time.perf_counter()
            _, _, st = oracle_api.render(env, width, height, time=args.time, threads=threads)
            return st["segments"], time.perf_counter() - t0, height, f"whole {width}x{height} frames"
        segs, secs, rows, d, _ = oracle_sample(env, width, height, args.time, n_blocks=9, rows_per_block=args.ref_rows, threads=threads)
        return segs, secs, rows, d

    # the driver's K and W also size the GPU arm, where a frame takes milliseconds: keep the CPU run within a few
    # minutes by shortening the warm-up first, then the timed frames (never below 3), and say so in the line
    steps, warmup = args.steps, args.warmup
    budget_s = 240.0
    _, probe_s, probe_rows, _ = one_step()
    frame_s = probe_s * (height / probe_rows)
    if whole and frame_s * (steps + warmup) > budget_s:
        warmup = 0
        steps = max(min(steps, 3), min(steps, int(budget_s / frame_s)))
    for _ in range(max(0, warmup - 1)):
        one_step()
    for _ in range(steps):
        segs, secs, rows, desc = one_step()
        seg_total += segs
        sec_total += secs
        rows_total += rows
    value = seg_total / sec_total / 1e6
    ms_frame = sec_total / steps * 1e3 * (height / (rows_total / steps))
    note = "whole frames: ms_per_step is measured" if whole else "ms_per_step extrapolated from the sampled rows to the full frame"
    if steps != args.steps:
        note += f"; {steps} timed frames instead of {args.steps} to bound the CPU run to ~{int(budget_s)} s"
    line = {
        "impl": "reference", "metric": "Mrays/s", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": ms_frame, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.scene} {width}x{height} max_depth {env.camera.max_depth} time {args.time}", "note": note},
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_RESULT_OUT = sys.stdout


def emit(obj) -> None:
    """The result lines go to the process's ORIGINAL stdout (see main)."""
    print(json.dumps(obj), file=_RESULT_OUT, flush=True)


class Rig:
    """One config (scene, frame size, depth) on this rank: device-resident steps, host-frame steps, teardown."""

    def __init__(self, args, scene, width, height, max_depth, world, rank, local_rank, precision="f64"):
        import torch
        import torch.distributed as dist

        import euclider_b200 as eb
        from euclider_b200 import bands

        self.torch, self.dist, self.eb = torch, dist, eb
        self.args, self.scene, self.width, self.height = args, scene, width, height
        self.world, self.rank, self.local_rank = world, rank, local_rank
        self.device = torch.device("cuda", local_rank)
        env = eb.load_reference_scene(scene)
        if max_depth:
            env.camera.max_depth = max_depth
        env.pipeline = eb.EUCL_PIPELINE_MEGAKERNEL if args.pipeline == "megakernel" else eb.EUCL_PIPELINE_WAVEFRONT
        env.precision = precision
        self.stream = torch.cuda.current_stream()
        env.set_stream(self.stream.cuda_stream, device=local_rank)
        self.env = env
        self.band_rows = args.band_rows if world > 1 else 0
        opts = eb.EuclRenderOpts(width=width, height=height, band_rows=self.band_rows, band_rank=rank, band_world=world)
        self.my_rows = int(eb.lib().eucl_band_rows_for_rank(opts)) if world > 1 else height
        self.frame_bytes = height * width * 3
        self.peer = world > 1 and args.gather == "peer"
        self.frame_ptr, self.frame, self.ipc_ptr = 0, None, None
        if world == 1:
            self.frame = torch.empty((height, width, 3), dtype=torch.uint8, device=self.device)
            self.frame_ptr = self.frame.data_ptr()
        elif self.peer:
            # One frame buffer on GPU 0, mapped into every rank through CUDA IPC: each rank's pack kernel
            # stores its rows straight into it over NVLink, so the gather IS the last kernel of the frame.
            handle = torch.zeros(eb._capi.EUCL_IPC_HANDLE_BYTES, dtype=torch.uint8, device=self.device)
            ptr = C.c_void_p()
            if rank == 0:
                eb._capi.check(eb.lib().eucl_device_malloc(local_rank, self.frame_bytes, C.byref(ptr)))
                buf = (C.c_uint8 * eb._capi.EUCL_IPC_HANDLE_BYTES)()
                eb._capi.check(eb.lib().eucl_ipc_export(ptr, buf))
                handle.copy_(torch.tensor(list(buf), dtype=torch.uint8))
            dist.broadcast(handle, src=0)
            if rank != 0:
                buf = (C.c_uint8 * eb._capi.EUCL_IPC_HANDLE_BYTES)(*handle.cpu().tolist())
                eb._capi.check(eb.lib().eucl_ipc_open(buf, local_rank, C.byref(ptr)))
            self.ipc_ptr = ptr
            self.frame_ptr = ptr.value
            if rank == 0:  # torch view of the raw allocation (for --check)
                fp = self.frame_ptr

                class _Raw:
                    __cuda_array_interface__ = {"shape": (height, width, 3), "typestr": "|u1", "data": (fp, False), "version": 2}
                self.frame = torch.as_tensor(_Raw(), device=self.device)
            # frame-complete flag: a stream-ordered all-reduce after each rank's last kernel; nothing blocks on the host
            self.flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        else:
            # NCCL gather of compact row blocks, scattered to frame rows on rank 0
            self.d_rows = torch.empty((max(self.my_rows, 1), width, 3), dtype=torch.uint8, device=self.device)
            self.frame = torch.empty((height, width, 3), dtype=torch.uint8, device=self.device) if rank == 0 else None
            self.rows_of = [torch.tensor(bands.local_rows(height, self.band_rows, r, world), dtype=torch.long, device=self.device)
                            for r in range(world)]
            max_rows = max(len(x) for x in self.rows_of)
            self.send = torch.zeros((max_rows, width, 3), dtype=torch.uint8, device=self.device)
            self.recv = [torch.empty_like(self.send) for _ in range(world)] if rank == 0 else None
        # host frame of the e2e leg: pinned; at N > 1 ONE frame in shared memory that every rank maps and pins
        self.shm_path, self.host_np, self.sync_np, self.host_pinned = None, None, None, False
        if world == 1:
            self.host = torch.empty((height, width, 3), dtype=torch.uint8).pin_memory()
            self.host_np = self.host.numpy()
            self.host_pinned = True
        else:
            name = [f"/dev/shm/eucl_bench_{os.getpid()}_{scene}_{width}x{height}"] if rank == 0 else [None]
            if rank == 0:
                with open(name[0], "wb") as f:
                    f.truncate(self.frame_bytes + 4096)
            dist.broadcast_object_list(name, src=0)
            self.shm_path = name[0]
            mm = np.memmap(self.shm_path, dtype=np.uint8, mode="r+", shape=(self.frame_bytes + 4096,))
            self.mm = mm
            self.host_np = mm[:self.frame_bytes].reshape(height, width, 3)
            self.sync_np = mm[self.frame_bytes:self.frame_bytes + 8 * world].view(np.int64)  # one arrival counter per rank
            self.host_pinned = eb.lib().eucl_host_register(C.c_void_p(mm.ctypes.data), mm.nbytes) == 0
            self.e2e_frames = 0
            dist.barrier()

    # -- the value leg: frame stays in HBM ---------------------------------------------------------
    def step(self, profile=False):
        a, env = self.args, self.env
        if self.world == 1 or self.peer:
            st = env.render_device(self.frame_ptr, (self.width, self.height), a.time, device=self.local_rank,
                                   band_rows=self.band_rows, band_rank=self.rank, band_world=self.world, compact_rows=False,
                                   profile=profile)
            if self.peer:  # the frame is complete when every rank's rows have landed: device-side, stream-ordered
                self.dist.all_reduce(self.flag)
            return st
        st = env.render_device(self.d_rows.data_ptr(), (self.width, self.height), a.time, device=self.local_rank,
                               band_rows=self.band_rows, band_rank=self.rank, band_world=self.world, compact_rows=True,
                               profile=profile)
        self.send[:self.my_rows].copy_(self.d_rows[:self.my_rows])
        self.dist.gather(self.send, self.recv, dst=0)
        if self.rank == 0:
            for r in range(self.world):
                self.frame.index_copy_(0, self.rows_of[r], self.recv[r][:len(self.rows_of[r])])
        return st

    # -- the e2e leg: the reference-facing call with a HOST frame ----------------------------------
    def e2e_step(self):
        a, env = self.args, self.env
        img = env.render((self.width, self.height), a.time, device=self.local_rank, out=self.host_np,
                         band_rows=self.band_rows, band_rank=self.rank, band_world=self.world)
        if self.world > 1:  # frame complete = every rank has copied its bands into the shared host frame
            self.e2e_frames += 1
            self.sync_np[self.rank] = self.e2e_frames
            while int(self.sync_np.min()) < self.e2e_frames:
                pass
        return img.stats

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def close(self):
        eb = self.eb
        self.sync_all()
        if self.shm_path is not None:
            if self.host_pinned:
                eb.lib().eucl_host_unregister(C.c_void_p(self.mm.ctypes.data))
            self.host_np = self.sync_np = None
            del self.mm
            self.dist.barrier()
            if self.rank == 0:
                try:
                    os.unlink(self.shm_path)
                except OSError:
                    pass
        self.env.set_stream(0, device=self.local_rank)
        self.frame = None
        if self.ipc_ptr is not None:
            if self.rank != 0:
                eb.lib().eucl_ipc_close(self.ipc_ptr)
            self.dist.barrier()
            if self.rank == 0:
                eb.lib().eucl_device_free(self.local_rank, self.ipc_ptr)
        self.env.close()
        self.torch.cuda.empty_cache()


def settle_frames(warmup: int) -> int:
    """Untimed frames in front of the timed region.  A scene settles in its first frames: the node arena grows to its
    size (frame 0), the ray-grouping mode is chosen from two frames of each setting (frames 1-4), the chosen launch
    sequence is seen once and captured as a CUDA graph (frames 5-6).  Fewer warm-up frames than that would time the
    tuner, not the renderer; the line reports the number actually used."""
    return max(warmup, 8)


DUMP_MAX_PIXELS = 1 << 21  # 24 MiB of float32 RGB, plus 16 MiB of float64 pixel indices when sampled


def dump_outputs(out_dir: str, frame, stats: dict) -> None:
    """Writes what the last timed step handed its caller: the RGB8 frame (row 0 = bottom) as float32 and the ray-tree
    node count of every level as float64.  A frame of more than DUMP_MAX_PIXELS pixels is sampled: the same
    seeded choice of pixels for the same frame size, their flat indices (y * width + x) in frame_pixel_index.npy."""
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    rgb = frame.cpu().numpy().reshape(-1, 3)
    if rgb.shape[0] > DUMP_MAX_PIXELS:
        index = np.sort(np.random.default_rng(0).choice(rgb.shape[0], DUMP_MAX_PIXELS, replace=False))
        rgb = rgb[index]
        np.save(out / "frame_pixel_index.npy", index.astype(np.float64))
    else:
        rgb = rgb.reshape(frame.shape)
    np.save(out / "frame.npy", rgb.astype(np.float32))
    np.save(out / "level_counts.npy", np.array(stats["level_counts"], dtype=np.float64))  # at N > 1: rank 0's rows


def measure(rig: Rig, steps: int, warmup: int, sample_clocks: bool, dump_dir: str | None = None):
    """Device-timed value leg, profile pass, e2e leg.  Returns a dict on rank 0, None elsewhere.
    With `dump_dir`, rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    torch, dist = rig.torch, rig.dist
    world, rank = rig.world, rig.rank
    for _ in range(settle_frames(warmup)):
        rig.step()
    rig.sync_all()
    sampler = ClockSampler(rig.local_rank) if (sample_clocks and rank == 0) else None
    if sampler:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    segs, launches, retries, own_ms, grouping = 0, 0, 0, 0.0, 0
    ev0.record(rig.stream)
    for _ in range(steps):
        st = rig.step()
        segs += st["segments"]
        launches += st["launches"]
        retries += st["retries"]
        own_ms += st["ms_total"]
        grouping = st["ray_grouping"]
    ev1.record(rig.stream)
    rig.sync_all()
    ms = ev0.elapsed_time(ev1)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, rig.frame, st)
    clocks = sampler.stop() if sampler else None
    prof = rig.step(profile=True)  # per-kernel-family device times (extra events; outside the timed region)
    rig.sync_all()
    t = torch.tensor([ms, float(segs), float(launches), float(retries), own_ms / steps, prof["ms_intersect"], float(prof["segments"])],
                     dtype=torch.float64, device=rig.device)
    if world > 1:
        allt = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        allt = torch.stack(allt).cpu().numpy()
    else:
        allt = t.cpu().numpy()[None, :]
    ms = float(allt[:, 0].max())
    segs, launches, retries = int(allt[:, 1].sum()), int(allt[:, 2].sum()), int(allt[:, 3].sum())
    # end to end: host frame, copies inside the timed region, wall clock between barriers
    for _ in range(4):  # another output buffer: its launch sequence is seen, captured, then replayed
        rig.e2e_step()
    rig.sync_all()
    t0 = time.perf_counter()
    e2e_segs = 0
    for _ in range(steps):
        e2e_segs += rig.e2e_step()["segments"]
    rig.sync_all()
    e2e_s = time.perf_counter() - t0
    tt = torch.tensor([e2e_s, float(e2e_segs)], dtype=torch.float64, device=rig.device)
    if world > 1:
        tm, ts = tt.clone(), tt.clone()
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dist.all_reduce(ts, op=dist.ReduceOp.SUM)
        e2e_s, e2e_segs = float(tm[0]), float(ts[1])
    if rank != 0:
        return None
    return {
        "ms_per_step": ms / steps, "value": segs / (ms * 1e-3) / 1e6, "segments_per_frame": segs / steps, "launches": launches,
        "retries": retries, "clocks": clocks, "ray_grouping": int(grouping), "prof": prof,
        "rank_ms": [round(float(v), 4) for v in allt[:, 4]],  # each rank's own device time per frame (CUDA events around its kernels)
        "k_intersect_ms_max": float(allt[:, 5].max()), "prof_segments": float(allt[:, 6].sum()),
        "e2e": {"value": e2e_segs / e2e_s / 1e6, "unit": "Mrays/s", "ms_per_step": e2e_s / steps * 1e3,
                "h2d_bytes_per_step": 256 * world, "d2h_bytes_per_step": rig.width * rig.height * 3,
                "host_frame": ("pinned" if rig.host_pinned else "pageable") + (", shared by all ranks (each copies its own bands)" if world > 1 else "")},
    }


def main():
    # stdout carries the JSON result lines and nothing else: libraries that write to file descriptor 1 on their own
    # (NCCL prints "NCCL version ..." there) are sent to stderr instead
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scene", default="3d_room")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--height", type=int, default=0)
    ap.add_argument("--time", type=float, default=0.0)
    ap.add_argument("--max-depth", type=int, default=0)
    ap.add_argument("--pipeline", default="wavefront", choices=["wavefront", "megakernel"])
    ap.add_argument("--band-rows", type=int, default=16)
    ap.add_argument("--ref-rows", type=int, default=None,
                    help="CPU legs: rows per sampled block (reference arm default 0 = whole frames; cpu_baseline default 32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the table of the other BASELINE.json configs")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N > 1: ranks store their rows into GPU 0's frame through CUDA IPC (peer) or NCCL gather")
    ap.add_argument("--check", action="store_true", help="N > 1: compare the gathered frames with a single-GPU render")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the frame and level counts of the last timed step as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    width, height = DEFAULT_CONFIGS.get(args.scene, (3840, 2160))
    width, height = args.width or width, args.height or height

    if args.impl == "reference":
        args.ref_rows = 0 if args.ref_rows is None else args.ref_rows
        run_reference(args, width, height)
        return
    args.ref_rows = 32 if args.ref_rows is None else args.ref_rows

    import torch
    import torch.distributed as dist

    import euclider_b200 as eb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)

    rig = Rig(args, args.scene, width, height, args.max_depth, world, rank, local_rank)
    m = measure(rig, args.steps, args.warmup, sample_clocks=True, dump_dir=args.dump_outputs)
    env = rig.env

    line = None
    if rank == 0:
        f_scene = scene_flops_per_segment(env)
        dadd, dmul, dfma = C.c_double(), C.c_double(), C.c_double()
        eb.lib().eucl_fp64_peak(local_rank, C.byref(dadd), C.byref(dmul), C.byref(dfma))
        peak = max(dadd.value, dmul.value)  # non-fused FP64 instruction rate, T op/s (-fmad=false build)
        achieved = m["prof_segments"] * f_scene / (m["k_intersect_ms_max"] * 1e-3) / 1e12 if m["k_intersect_ms_max"] > 0 else None
        roofline = {
            "bound": "fp64_issue", "unit": "Tflop/s", "peak": peak * world,
            "peak_source": f"measured live (DADD/DMUL microbenchmark on rank 0) x {world} GPU(s)", "peak_dfma_tops": dfma.value,
            "traffic": None, "traffic_note": "not measured in this run; dram__bytes of the kernels are in the ncu captures under profiles/",
            "flops_per_segment": f_scene, "kernel": "k_intersect, light + heavy build, all levels of one frame (slowest rank)",
            "achieved": achieved, "frac": achieved / (peak * world) if achieved else None, "kernel_ms_per_frame": m["k_intersect_ms_max"],
            "family_ms": {k: m["prof"][k] for k in ("ms_raygen", "ms_intersect", "ms_shade", "ms_resolve", "ms_total")},
            # the timed frames run two pipelines side by side (EUCL_SPLIT); the profile frame runs the same launches one after
            # the other with an event after each, so its family times add up to more than ms_per_step and `frac` is the
            # kernels' rate when timed alone, launch by launch
            "kernel_share_of_profile_frame": m["prof"]["ms_intersect"] / max(1e-9, sum(m["prof"][k] for k in ("ms_raygen", "ms_intersect", "ms_shade", "ms_resolve"))),
        }
        cpu = None
        if not args.no_cpu_baseline and world == 1:  # reported at N = 1 only
            try:
                c_segs, c_secs, _, desc, threads = oracle_sample(env, width, height, args.time, rows_per_block=args.ref_rows)
                cpu = {"value": c_segs / c_secs / 1e6, "unit": "Mrays/s", "cores": threads, "kind": "port", "sample": desc}
            except Exception as exc:  # the oracle is test infrastructure; its absence must not hide the GPU number
                cpu = {"value": None, "unit": "Mrays/s", "cores": 0, "kind": "port", "sample": f"unavailable: {exc}"}
        line = {
            "metric": "Mrays/s", "value": m["value"], "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": settle_frames(args.warmup), "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.scene} {width}x{height} max_depth {env.camera.max_depth} time {args.time}",
                       "pipeline": args.pipeline, "segments_per_frame": m["segments_per_frame"],
                       "ray_grouping": m["ray_grouping"],  # what the per-scene tuner settled on (EuclStats.ray_grouping)
                       "parallelism": (f"row bands of {rig.band_rows} x {world} ranks, "
                                       + ("peer stores into GPU 0's frame (CUDA IPC over NVLink), frame-complete flag = "
                                          "stream-ordered all-reduce" if rig.peer else "NCCL gather to rank 0"))
                       if world > 1 else "single GPU",
                       "pipelines_per_frame": int(os.environ.get("EUCL_SPLIT", "2")),  # concurrent pipelines per rank (render_split)
                       "l2": "node arena (GBs per chunk) is far larger than the 126 MB L2; no explicit flush"},
            "fps": 1e3 / m["ms_per_step"], "e2e": m["e2e"], "gpu_launches": m["launches"], "retries": m["retries"],
            "clocks": m["clocks"], "rank_device_ms": {"min": min(m["rank_ms"]), "max": max(m["rank_ms"]), "per_rank": m["rank_ms"]},
            "roofline": roofline, "cpu_baseline": cpu,
        }
    check_results = []
    if world > 1 and args.check:
        check_results.append(check_gather(rig, args))
    rig.close()

    # the other configs of BASELINE.json, same run, fewer frames each
    if not args.no_configs and args.pipeline == "wavefront":
        table = []
        todo = ALL_CONFIGS if world == 1 else MULTI_GPU_CONFIGS
        k = max(3, min(args.steps, 6))
        for scene, w, h, depth, precision in todo:
            r2 = Rig(args, scene, w, h, depth, world, rank, local_rank, precision)
            m2 = measure(r2, k, 3, sample_clocks=False)
            if rank == 0:
                f2 = scene_flops_per_segment(r2.env)
                ach = m2["prof_segments"] * f2 / (m2["k_intersect_ms_max"] * 1e-3) / 1e12 if m2["k_intersect_ms_max"] > 0 else None
                table.append({"scene": scene, "width": w, "height": h, "max_depth": int(r2.env.camera.max_depth), "dtype": precision,
                              "steps": k,
                              "ms_per_step": m2["ms_per_step"], "fps": 1e3 / m2["ms_per_step"], "mrays_per_s": m2["value"],
                              "segments_per_frame": m2["segments_per_frame"], "e2e_mrays_per_s": m2["e2e"]["value"],
                              "e2e_ms_per_step": m2["e2e"]["ms_per_step"], "flops_per_segment": f2,
                              # fraction of the f64 issue peak; f32 rows run on the FP32 pipes (twice the lanes): not comparable
                              "k_intersect_frac": (ach / (peak * world) if ach else None) if precision == "f64" else None,
                              "ray_grouping": m2["ray_grouping"],
                              "retries": m2["retries"], "rank_device_ms": [min(m2["rank_ms"]), max(m2["rank_ms"])]})
            if world > 1 and args.check:
                check_results.append(check_gather(r2, args))
            r2.close()
        if rank == 0:
            line["configs"] = table
    if rank == 0:
        emit(line)
        for c in check_results:
            emit(c)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def check_gather(rig: Rig, args):
    """N > 1: the gathered device frame and the shared host frame against a single-GPU render on rank 0."""
    rig.step()
    rig.e2e_step()
    rig.sync_all()
    res = None
    if rig.rank == 0:
        gathered = rig.frame.cpu().numpy()
        shared = np.array(rig.host_np)
        rig.env.set_stream(0, device=rig.local_rank)
        whole = rig.env.render((rig.width, rig.height), args.time, device=rig.local_rank)
        rig.env.set_stream(rig.stream.cuda_stream, device=rig.local_rank)
        res = {"check": f"{rig.scene} {rig.width}x{rig.height}: gathered frames == single-GPU frame",
               "device_frame_equal": bool(np.array_equal(whole.data, gathered)),
               "host_frame_equal": bool(np.array_equal(whole.data, shared))}
    rig.sync_all()
    return res


if __name__ == "__main__":
    main()
