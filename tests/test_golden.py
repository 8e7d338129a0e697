"""Both oracle builds against the committed fixtures in tests/golden (made by tools/make_golden.py).

The Rust reference cannot be executed here, so these fixtures are oracle outputs frozen at the
commit that introduced them: they pin the oracle (and the scene front end feeding it) against
accidental change.  The GPU suite (test_parity_gpu.py) compares the CUDA path with the same files."""
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb

GOLDEN = sorted((Path(__file__).resolve().parent / "golden").glob("*.npz"))


@pytest.mark.parametrize("path", GOLDEN, ids=lambda p: p.stem)
@pytest.mark.parametrize("variant", ["det", "glibc"])
def test_oracle_matches_golden(oracle, path, variant):
    g = np.load(path)
    name = path.stem.rsplit("_", 1)[0]
    env = eb.load_reference_scene(name)
    rgb, hit, st = oracle.render(env, int(g["width"]), int(g["height"]), time=float(g["time"]), variant=variant)
    assert np.array_equal(hit.astype(np.int8), g[f"hit_{variant}"])
    assert st["level_counts"] == g[f"levels_{variant}"].tolist()
    assert np.array_equal(rgb, g[f"rgb_{variant}"])


@pytest.mark.parametrize("path", GOLDEN, ids=lambda p: p.stem)
def test_libm_choice_stays_inside_the_tolerance(path):
    """glibc vs deterministic libm: identical hit maps, every pixel within 1/255 (the north-star
    tolerance is >= 99.5 % of pixels within 1/255)."""
    g = np.load(path)
    assert np.array_equal(g["hit_det"], g["hit_glibc"])
    diff = np.abs(g["rgb_det"].astype(np.int16) - g["rgb_glibc"].astype(np.int16)).max(axis=-1)
    assert (diff <= 1).mean() >= 0.995
