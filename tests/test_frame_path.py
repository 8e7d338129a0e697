"""The ray-grouping tuner of the frame path (api_device.cu: choose_grouping, tune_grouping).  A fresh scene renders its
frames alternately with and without grouping by reach key, "on" first.  Only retry-free frames count, and never the
scene's very first frame.  Once each setting has two counted frames the faster one is kept.  No CUDA graph is captured
while the scene is still choosing, so capture time never distorts the comparison.  A frame split into two pipelines is
judged as a whole and follows the same schedule as one pipeline."""
import pytest

import euclider_b200 as eb

pytestmark = pytest.mark.gpu


def expected_schedule(retries):
    """Per frame: (ray grouping on, still choosing) as the documented schedule gives it for these retry counts."""
    counted = [0, 0]  # counted frames without / with grouping
    schedule = []
    for frame, r in enumerate(retries):
        choosing = min(counted) < 2
        on = counted[1] <= counted[0]
        if choosing and frame > 0 and r == 0:
            counted[int(on)] += 1
        schedule.append((on, choosing))
    return schedule


@pytest.mark.parametrize("split", [1, 2])
def test_ray_grouping_schedule(built_lib, monkeypatch, split):
    monkeypatch.delenv("EUCL_BIN_RAYS", raising=False)
    monkeypatch.setenv("EUCL_SPLIT_MIN_PIXELS", "0")
    monkeypatch.setenv("EUCL_SPLIT", str(split))
    env = eb.load_reference_scene("3d_room")
    stats = [env.render((256, 160)).stats for _ in range(8)]
    retries = [st["retries"] for st in stats]
    grouping = [st["ray_grouping"] for st in stats]
    replays = [st["graph_replays"] for st in stats]
    schedule = expected_schedule(retries)
    # (a frame with retries may trim its workspace, lists included, and then reports no grouping)
    for frame, (on, choosing) in enumerate(schedule):
        if choosing:
            assert replays[frame] == 0, (frame, retries, replays)
            if retries[frame] == 0:
                assert grouping[frame] == int(on), (frame, retries, grouping)
    kept = [grouping[frame] for frame, (_, choosing) in enumerate(schedule) if not choosing and retries[frame] == 0]
    assert len(set(kept)) <= 1, (retries, grouping)  # once chosen, the setting stays
