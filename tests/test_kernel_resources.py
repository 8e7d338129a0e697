"""The kernel builds a render without AOVs runs keep their registers, stack, local memory and shared memory: the AOV
builds (k_aov_primary, k_resolve_cost, k_final_cost, k_megakernel_aov) are kernels of their own, so asking for nothing
costs nothing.  tests/golden/kernel_resources.json pins those builds as `cuobjdump --dump-resource-usage` reports them
for the CUDA 12.9 toolkit; a kernel changed on purpose updates its entry there."""
import json
import re
import shutil
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden" / "kernel_resources.json"
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def resource_usage(path) -> dict:
    """Kernel -> {REG, STACK, LOCAL, SHARED}; the anonymous namespace's per-build tag is replaced by ANON."""
    out = subprocess.run([CUOBJDUMP, "--dump-resource-usage", str(path)], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            name = re.sub(r"\d+_GLOBAL__N__[0-9a-f]+_\d+_kernels_cu_[0-9a-f]+", "ANON", m.group(1))
        elif name and "REG:" in line:
            kv = dict(x.split(":", 1) for x in line.split())
            res[name] = {k: int(kv[k]) for k in ("REG", "STACK", "LOCAL", "SHARED")}
            name = None
    return res


def toolkit_version() -> str:
    out = subprocess.run([CUOBJDUMP, "--version"], capture_output=True, text=True).stdout
    m = re.search(r"release (\d+\.\d+)", out)
    return m.group(1) if m else ""


@pytest.mark.skipif(not Path(CUOBJDUMP).exists(), reason="cuobjdump (CUDA toolkit) not installed")
def test_plain_kernel_builds_keep_their_resources(built_lib):
    from euclider_b200 import _capi

    golden = json.loads(GOLDEN.read_text())
    if toolkit_version() != golden["toolkit"]:
        pytest.skip(f"resources are pinned for CUDA {golden['toolkit']}")
    now = resource_usage(_capi.LIB_PATH)
    changed = {k: (v, now.get(k)) for k, v in golden["kernels"].items() if now.get(k) != v}
    assert not changed, f"kernel builds changed (pinned, now): {changed}"
    new = sorted(k for k in now if k not in golden["kernels"])
    for tag in ("k_aov_primary", "k_resolve_cost", "k_final_cost", "k_megakernel_aov"):
        assert any(tag in k for k in new), f"{tag} is missing from the library"
