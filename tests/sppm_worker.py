"""Worker of tests/test_sppm_multi_gpu.py (launched by torch.distributed.run, one process per GPU): a sharded SPPM render, with the library's
own communicator (`native`: cgrt_allgather_hitpoints and the all-reduce inside cgrt_round_update) or with host-driven collectives (`host`:
torch all_gather of the records, cgrt_import_hitpoints_dev, torch all_reduce of the accumulators on the library's stream). Checked on rank 0
against the same rounds on one GPU; every rank checks that its device memory reaches a steady state."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist

    from cgraytracing_b200 import Context, RenderConfig, preset
    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer, make_native_comm

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    accum, how = int(sys.argv[1]), sys.argv[2]
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    W, H, ROUNDS, PER, LONG = 160, 120, 4, 50001, 31
    JITTER = 1
    cfg = RenderConfig(width=W, height=H, into_rule=1, update_mode=1)
    scene = preset("c2_bunny_chess")
    comm = make_native_comm(local, rank, world) if how == "native" else None
    free = {}
    with Context(local) as g:
        g.set_config(cfg, accum_mode=accum)
        scene.build_into(g); g.commit()
        R = ShardedRenderer(GpuEngine(g, local, comm, world, rank=rank, sppm=JITTER), rank, world)
        for r in range(LONG):
            R.eye(H)
            R.round(PER)
            if r == ROUNDS - 1:
                px = g.sppm_download_pixels()
                img = g.gather_image(float(ROUNDS * PER))
            if r in (3, 30):
                g.synchronize()
                torch.cuda.synchronize(local)
                free[r] = torch.cuda.mem_get_info(local)[0]
        if comm is not None:
            g.set_comm(0, 1)
    # every rank holds the same pixels
    t = torch.tensor([float(px["n"].sum()), float(px["tau"].sum()), float(img.sum())], device=f"cuda:{local}", dtype=torch.float64)
    lo, hi = t.clone(), t.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN); dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    assert torch.equal(lo, hi), (lo, hi)
    # device memory: the per-round buffers (tiles, gathered records, grid) come back at the same sizes
    assert abs(free[3] - free[30]) <= 64 << 20, (rank, (free[3] - free[30]) / 2**20)
    if rank == 0:
        with Context(local) as s:
            s.set_config(cfg, accum_mode=accum)
            scene.build_into(s); s.commit(); s.set_sppm(JITTER)
            for r in range(ROUNDS):
                s.sppm_begin_round(r); s.photon_pass(r * PER, PER); s.round_update()
            ref = s.sppm_download_pixels()
            rimg = s.gather_image(float(ROUNDS * PER))
        assert np.array_equal(px["n"], ref["n"]) and px["n"].sum() > 0  # accepted photons per pixel: equal
        assert np.array_equal(px["r2"], ref["r2"])                      # hence the same radii, bit for bit
        tol = 1e-9 if accum == 0 else 1e-4
        assert np.allclose(px["tau"], ref["tau"], rtol=tol, atol=1e-12)
        assert np.allclose(img, rimg, rtol=tol, atol=1e-12)
        print("SPPM_OK", how, accum, int(px["n"].sum()))
    dist.barrier()
    if comm is not None:
        from cgraytracing_b200.binding import comm_destroy

        comm_destroy(comm)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
