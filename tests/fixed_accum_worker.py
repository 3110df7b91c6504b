"""Worker of tests/test_fixed_accum.py.

  fixed_accum_worker.py guard OUT.npz   one c3 render in accum_mode 2 (run with CGRT_GUARD=1): its observables and the damaged fence bytes
  fixed_accum_worker.py ranks HOW       (torch.distributed.run, one process per GPU) a sharded accum_mode 2 render whose round exchange is
                                        HOW = nccl (the library's communicator), peer (peer memory) or torch (torch.distributed all-reduce of
                                        the int64 accumulators); rank 0 checks it against one GPU bit for bit."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def guard(out):
    import cgraytracing_b200 as cg
    from tests import test_fixed_accum as t

    scene, cfg = t.case("c3")
    with t.gpu_context(cg, scene, cfg, t.PPM) as g:
        g.eye_pass()
        g.build_grid()
        for r in range(t.ROUNDS):
            for first, count in ((r * t.PHOTONS, t.PHOTONS // 3), (r * t.PHOTONS + t.PHOTONS // 3, t.PHOTONS - t.PHOTONS // 3)):
                g.photon_pass(first, count)
            g.round_update()
        _, rgb8 = g.gather_image(float(t.ROUNDS * t.PHOTONS), want_rgb8=True)
        o = t.observables(g, t.PPM, float(t.ROUNDS * t.PHOTONS), rgb8)
        damaged = g.check_guards()
    np.savez(out, damaged=np.int64(damaged), **o)


def ranks(how):
    import torch
    import torch.distributed as dist

    from cgraytracing_b200 import Context
    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer, make_native_comm
    from tests import test_fixed_accum as t

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    scene, cfg = t.case("c2")
    rounds, per = 4, 50001
    comm = make_native_comm(local, rank, world) if how in ("nccl", "peer") else None
    with Context(local) as g:
        g.set_config(cfg, accum_mode=2)
        scene.build_into(g)
        g.commit()
        R = ShardedRenderer(GpuEngine(g, local, comm, world, rank=rank, peer=(how == "peer")), rank, world)
        R.render(cfg.height, rounds, per)
        _, rgb8 = g.gather_image(float(rounds * per), want_rgb8=True)
        got = t.observables(g, t.PPM, float(rounds * per), rgb8)
    if rank == 0:
        with Context(local) as s:
            s.set_config(cfg, accum_mode=2)
            scene.build_into(s)
            s.commit()
            s.eye_pass()
            s.build_grid()
            for r in range(rounds):
                s.photon_pass(r * per, per)
                s.round_update()
            _, rgb8 = s.gather_image(float(rounds * per), want_rgb8=True)
            one = t.observables(s, t.PPM, float(rounds * per), rgb8)
        assert got["n"].sum() > 0
        t.assert_same(got, one)
        print("FIXED_RANKS_OK", how, int(got["n"].sum()), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    if sys.argv[1] == "guard":
        guard(sys.argv[2])
    else:
        ranks(sys.argv[2])
