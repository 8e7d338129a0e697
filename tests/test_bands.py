"""Row-band sharding: host logic, C library agreement, and a world_size-2 gloo run on CPU in which
each rank renders its bands (with the CPU oracle standing in for the device) and rank 0 gathers."""
import os
import socket
import sys
from pathlib import Path

import numpy as np
import pytest

import euclider_b200 as eb
from euclider_b200 import bands

ROOT = Path(__file__).resolve().parent.parent


@pytest.mark.parametrize("height,band,world", [(54, 8, 2), (54, 16, 4), (7, 3, 8), (2160, 16, 8), (10, 0, 1), (5, 8, 2)])
def test_partition_is_exact(built_lib, height, band, world):
    seen = []
    for r in range(world):
        rows = bands.local_rows(height, band, r, world)
        opts = eb.EuclRenderOpts(width=4, height=height, band_rows=band, band_rank=r, band_world=world)
        assert built_lib.eucl_band_rows_for_rank(opts) == len(rows)
        seen += rows
    assert sorted(seen) == list(range(height))


def _worker(rank, world, port, height, width, band, q):
    sys.path.insert(0, str(ROOT))
    sys.path.insert(0, str(ROOT / "tests"))
    import torch
    import torch.distributed as dist

    import oracle_api

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    env = eb.load_reference_scene("3d_fresnel")
    rows = bands.local_rows(height, band, rank, world)
    mine = np.zeros((len(rows), width, 3), np.uint8)
    for k, y in enumerate(rows):  # the oracle renders one frame row at a time
        mine[k] = oracle_api.render(env, width, height, threads=1, rows=(y, y + 1))[0][0]
    max_rows = max(len(bands.local_rows(height, band, r, world)) for r in range(world))
    send = torch.zeros((max_rows, width, 3), dtype=torch.uint8)
    send[:len(rows)] = torch.from_numpy(mine)
    recv = [torch.empty_like(send) for _ in range(world)] if rank == 0 else None
    dist.gather(send, recv, dst=0)
    if rank == 0:
        frame = bands.gather_frame([r.numpy() for r in recv], height, band, world)
        q.put(frame)
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gather_gloo(oracle):
    import torch.multiprocessing as mp

    height, width, band, world = 27, 48, 4, 2
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, height, width, band, q)) for r in range(world)]
    for p in procs:
        p.start()
    frame = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    env = eb.load_reference_scene("3d_fresnel")
    whole = oracle.render(env, width, height)[0]
    assert np.array_equal(frame, whole)


def test_sub_pipelines_partition_a_ranks_rows():
    """render_split hands pipeline p of k the bands of rank `rank + p * world` in a world of `k * world`: together they
    are exactly the rank's rows, for ragged heights too."""
    lib = eb.lib()
    for height in (1, 16, 31, 32, 67, 131, 2160):
        for band in (4, 16):
            for world in (1, 2, 3, 8):
                for rank in range(world):
                    whole = eb.EuclRenderOpts(width=4, height=height, band_rows=band, band_rank=rank, band_world=world)
                    for k in (2, 3):
                        parts = 0
                        for p in range(k):
                            sub = eb.EuclRenderOpts(width=4, height=height, band_rows=band, band_rank=rank + p * world,
                                                    band_world=k * world)
                            parts += lib.eucl_band_rows_for_rank(sub)
                        assert parts == lib.eucl_band_rows_for_rank(whole), (height, band, world, rank, k)
