"""The dynamic shared-memory limit a scene sets on its kernels is process-wide: every scene launches the same kernels.  A
scene created later with smaller tables must not lower it below what an earlier, larger scene launches with.

A scene's heavy kernels (k_intersect, the megakernel) take the staged scene blob plus 32 KB of plane-chain scratch
(kPlaneChainMax doubles for each of kBlock threads), so a blob above 16 KB puts them over the 48 KB a kernel gets without
opting in.  The blob is what BlobWriter packs in eucl_scene_create (api_device.cu); `blob_lower_bound` adds up the
primitive tables alone, so it never overestimates."""
import json
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb

pytestmark = pytest.mark.gpu

PARSER = eb.Parser.default(resource_root=Path(__file__).resolve().parent.parent)
OPT_IN_FREE = 16 * 1024  # blob bytes that fit the 48 KB default next to the 32 KB scratch


def align16(n):
    return (n + 15) & ~15


def blob_lower_bound(n_prims, max_dim=4, plane_stride=6):
    """BlobWriter's primitive tables: kind (int32), v0 and v1 (double[max_dim] each, one plane per component), s0 and s1
    (double), and the AoS plane records (plane_stride doubles); each table starts on a 16-byte boundary."""
    return (align16(4 * n_prims) + 2 * align16(8 * max_dim * n_prims) + 2 * align16(8 * n_prims)
            + align16(8 * plane_stride * n_prims))


def spheres_scene(n):
    """A Void3 around the camera and `n` small spheres in a grid in front of it, every third a half mirror."""
    entities = []
    for i in range(n):
        y, z = (i % 20 - 9.5) * 0.5, (i // 20 - 5) * 0.5
        surface = {"ComposableSurface3": {
            "reflection_ratio": {"reflection_ratio_uniform_3": [0.5 if i % 3 == 0 else 0.0]},
            "reflection_direction": {"reflection_direction_specular_3": []},
            "threshold_direction": {"threshold_direction_identity_3": []},
            "surface_color": {"surface_color_uniform_3": [{"Rgba::new": [(i % 7) / 7, (i % 5) / 5, (i % 3) / 3, 1.0]}]}}}
        entities.append({"Entity3Impl::new": [{"Sphere3::new": [{"Point3::new": [10 + (i % 4), y, z]}, 0.2]},
                                              {"Vacuum3::new": []}, surface]})
    entities.append({"Void3::new_with_vacuum": []})
    return json.dumps({"Universe3": {
        "camera": {"PitchYawCamera3": []},
        "entities": entities,
        "background": {"MappedTextureImpl3::new": [{"uv_sphere_3": [{"Point3::new": [0, 0, 0]}]},
                                                   {"texture_image_linear": ["./tests/scenes/checker_rgba.png"]}]}}})


def test_a_smaller_scene_does_not_lower_the_shared_memory_limit(built_lib, oracle):
    large, small = PARSER.parse(spheres_scene(200)), PARSER.parse(spheres_scene(140))
    # both above the 48 KB default; `small` has the same tables for fewer spheres, so its blob is smaller
    assert blob_lower_bound(small.flat.n_prims) > OPT_IN_FREE
    assert small.flat.n_prims < large.flat.n_prims
    large._device_scene(0)  # created first: opts its kernels in to its shared memory
    small._device_scene(0)  # created last: configures the same kernels for its own, smaller size
    w, h = 96, 64
    img = large.render((w, h), time=0.5, want_hit_ids=True)
    rgb, hit, st = oracle.render(large, w, h, time=0.5, variant="det")
    assert np.array_equal(img.data, rgb)
    assert np.array_equal(img.hit_ids, hit)
    assert img.stats["segments"] == st["segments"]
    assert len(np.unique(hit)) > 20  # the frame shows many of the spheres
