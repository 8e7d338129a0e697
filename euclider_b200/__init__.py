"""euclider_b200 -- B200-native (sm_100a) renderer for euclider's per-pixel trace loop.

Public surface = the reference's interface for this path: `Parser` (scene JSON -> Environment)
and `Environment.render` (one RGB8 frame), backed by libeuclider_b200.so (C ABI, see
include/euclider_b200.h).  No CPU rendering fallback exists in this package.
"""
from pathlib import Path

from ._capi import EuclAovs, EuclCamera, EuclError, EuclFrame, EuclRays, EuclRenderOpts, EuclStats, EUCL_PIPELINE_MEGAKERNEL, EUCL_PIPELINE_WAVEFRONT, lib
from .scene import (AOV_NAMES, TREE_NODE_DTYPE, Environment, Parser, ParserError, RawFrames, RawImage2d, RawRays, RayTree,
                    SimulationContext, camera_step, default_tree_capacity, equirect_rays)

ROOT = Path(__file__).resolve().parent.parent
ASSET_ROOT = ROOT / "assets"  # the reference scenes, restated, and stand-in textures (assets/make_assets.py)


def load_reference_scene(name: str) -> Environment:
    """Parses assets/scenes/<name>.json with textures resolved under assets/."""
    return Parser.default(resource_root=ASSET_ROOT).parse_file(ASSET_ROOT / "scenes" / f"{name}.json")


__all__ = ["Parser", "Environment", "SimulationContext", "RawImage2d", "RawFrames", "RawRays", "EuclFrame", "EuclAovs", "EuclRays", "equirect_rays", "camera_step", "AOV_NAMES", "RayTree", "TREE_NODE_DTYPE", "default_tree_capacity", "ParserError", "EuclError", "EuclCamera",
           "EuclRenderOpts", "EuclStats", "EUCL_PIPELINE_WAVEFRONT", "EUCL_PIPELINE_MEGAKERNEL", "lib",
           "load_reference_scene", "ASSET_ROOT", "ROOT"]
