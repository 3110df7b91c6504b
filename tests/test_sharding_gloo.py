"""CPU, world_size 2, gloo: the host-side multi-GPU logic of cgraytracing_b200/distributed.py (row tiles for the eye pass +
all-gather of hitpoint records, disjoint photon index ranges, one all-reduce of the accumulators per round). The engine
behind the protocol is the CPU oracle here (tests only); on the GPU box the same class drives `GpuEngine`."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from cgraytracing_b200 import RenderConfig, preset
from cgraytracing_b200.distributed import ShardedRenderer, photon_shard, row_shard, split_range
from tests.util import OracleEngine

W, H, ROUNDS, PHOTONS = 64, 48, 2, 5001  # odd photon count: the remainder path


def test_split_range_is_disjoint_and_covering():
    for first, count, world in ((0, 10, 3), (7, 0, 2), (5, 1, 4), (0, 16 << 20, 8), (123, 1000003, 7)):
        parts = [split_range(first, count, r, world) for r in range(world)]
        assert parts[0][0] == first and sum(n for _, n in parts) == count
        for (a, n), (b, _) in zip(parts, parts[1:]):
            assert a + n == b
        assert max(n for _, n in parts) - min(n for _, n in parts) <= 1
    assert photon_shard(3, 1000, 1, 4) == (3250, 250)
    assert [row_shard(1024, r, 8) for r in (0, 7)] == [(0, 128), (896, 1024)]
    assert [row_shard(5, r, 8)[1] - row_shard(5, r, 8)[0] for r in range(8)] == [1, 1, 1, 1, 1, 0, 0, 0]
    with pytest.raises(ValueError):
        split_range(0, 10, 2, 2)


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = RenderConfig(width=W, height=H, update_mode=1, into_rule=1)
        eng = OracleEngine(preset("c2_bunny_chess"), cfg)
        r = ShardedRenderer(eng, rank, world)
        img = r.render(H, ROUNDS, PHOTONS)
        hp = eng.o.download_hitpoints()
        np.savez(os.path.join(out, f"rank{rank}.npz"), img=img, n=hp["n"], r2=hp["r2"], flux=hp["flux"], key=hp["key"], pos=hp["pos"])
    finally:
        dist.destroy_process_group()


def test_two_ranks_equal_one_rank(tmp_path):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    # single-rank run of the same job
    cfg = RenderConfig(width=W, height=H, update_mode=1, into_rule=1)
    eng = OracleEngine(preset("c2_bunny_chess"), cfg)
    img1 = ShardedRenderer(eng).render(H, ROUNDS, PHOTONS)
    hp1 = eng.o.download_hitpoints()
    for k in ("img", "n", "r2", "flux", "key", "pos"):  # replicas stay bit-identical
        assert np.array_equal(a[k], b[k]), k
    # the tile-sharded eye pass + all-gather reproduces the canonical hitpoint order exactly
    assert np.array_equal(a["key"], hp1["key"]) and np.array_equal(a["pos"], hp1["pos"])
    # integer counts exact; sums differ only by fp64 association (two partial sums added by the all-reduce)
    assert np.array_equal(a["n"], hp1["n"]) and a["n"].sum() > 1000
    assert np.array_equal(a["r2"], hp1["r2"])
    assert np.allclose(a["flux"], hp1["flux"], rtol=1e-12, atol=1e-12)
    assert np.allclose(a["img"], img1, rtol=1e-12, atol=1e-14)
