#!/usr/bin/env python
"""Generates tests/golden/*.npz: small frames of every reference scene rendered by the CPU oracle.

The reference itself cannot run here (no Rust toolchain), so these fixtures pin the ORACLE (and,
through the GPU parity tests, the CUDA path) against regressions; they are not outputs of the
Rust binary.  Renders the scenes under assets/ (assets/make_assets.py).  Run from the repo root:
    python tools/make_golden.py
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import euclider_b200 as eb  # noqa: E402
import oracle_api  # noqa: E402

SCENES = ["3d_fresnel", "3d_room", "3d_hallways", "4d_frame", "4d_cylinders", "4d_room", "3d_frame", "3d_fresnel_2",
          "3d_photo", "4d_fresnel"]
W, H, T = 96, 54, 1.234


def main():
    out = ROOT / "tests" / "golden"
    out.mkdir(parents=True, exist_ok=True)
    for name in SCENES:
        env = eb.load_reference_scene(name)
        data = {}
        for variant in ("det", "glibc"):
            rgb, hit, st = oracle_api.render(env, W, H, time=T, variant=variant)
            data[f"rgb_{variant}"] = rgb
            data[f"hit_{variant}"] = hit.astype(np.int8)
            data[f"levels_{variant}"] = np.array(st["level_counts"], dtype=np.int64)
        np.savez_compressed(out / f"{name}_{W}x{H}.npz", width=W, height=H, time=T, **data)
        print(name, "segments", int(data["levels_det"][:-1].sum()))


if __name__ == "__main__":
    main()
