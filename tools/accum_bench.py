"""Photon-round throughput of the three accumulator modes (accum_mode 1 float, 2 fixed point, 0 fp64) on the BASELINE workloads c1-c5.

One GPU: for every workload the modes run alternately (1, 2, 0, 1, 2, 0, ...), --runs times each. A run builds its own context (eye pass
and grid untimed), warms up, then times --steps rounds (photon pass + round update) between CUDA events on the library's stream:
photons/s = photons per round * steps / elapsed. The deposit kernel's time per round (cgrt_get_timings slot 3) comes from a separate
round with profiling on, after the timed window. The card's name and power limit are read in the same process.

Launched by torch.distributed.run with 2 or more processes it measures c3 weak scaling instead (the same photons per GPU, rounds sharded
by cgraytracing_b200.distributed.ShardedRenderer over the library's communicator), mode 2 against mode 1.

  python tools/accum_bench.py --out profiles/r06_accum_modes_1gpu.json
  python -m torch.distributed.run --nproc-per-node 8 tools/accum_bench.py --out profiles/r06_accum_modes_8gpu.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (the workload table)

MODES = (1, 2, 0)
MODE_NAMES = {0: "fp64", 1: "float", 2: "fixed"}
# warm-up and timed rounds per workload: c5 is 1 Gi photons per round
STEPS = {"c1_spheres_bezier": (3, 20), "c2_bunny_chess": (3, 10), "c3_dragon_glass": (2, 8), "c4_bump_dof": (2, 8), "c5_dragon_4096": (1, 2)}


def card(device):
    """Name and power limit of the card, as nvidia-smi reports them (read only)."""
    q = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    parts = [p.strip() for p in q.stdout.strip().split(",")] if q.returncode == 0 else []
    return dict(zip(("name", "power_limit", "max_sm_clock"), parts)) if len(parts) == 3 else {"nvidia_smi": q.stderr.strip()}


def config(name):
    from cgraytracing_b200 import RenderConfig, preset

    bench.select_workload(name)
    return preset(bench.PRESET), bench.make_config(RenderConfig), bench.PHOTONS_PER_ROUND


def one_run(device, name, mode, warmup, steps):
    import torch

    from cgraytracing_b200 import Context

    scene, cfg, P = config(name)
    with Context(device) as g:
        g.set_config(cfg, accum_mode=mode)
        scene.build_into(g)
        g.commit()
        g.eye_pass()
        g.build_grid()
        r = 0
        for _ in range(warmup):
            g.photon_pass(r * P, P); g.round_update(); r += 1
        g.synchronize()
        stream = torch.cuda.ExternalStream(g.stream())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            g.photon_pass(r * P, P); g.round_update(); r += 1
        g.accum_dev()  # the last round's update runs on the library's side stream: make the timed stream wait for it
        e1.record(stream)
        g.synchronize()
        ms = e0.elapsed_time(e1)
        g.set_profiling(True)
        before = g.timings()["photon_deposit"]
        g.photon_pass(r * P, P); g.round_update()
        g.synchronize()
        dep = g.timings()["photon_deposit"] - before
        n = int(g.download_hitpoints(fields=("n",))["n"].sum())
    return dict(mode=mode, ms_per_round=ms / steps, photons_per_s=P * steps / (ms * 1e-3), deposit_ms=dep, accepted_total=n)


def single_gpu(args):
    import torch

    out = dict(tool="tools/accum_bench.py", card=card(args.device), torch=torch.__version__, runs=args.runs, workloads={})
    for name in args.workloads:
        warmup, steps = STEPS[name]
        res = []
        for k in range(args.runs):
            for mode in MODES:
                t0 = time.time()
                r = one_run(args.device, name, mode, warmup, steps)
                r["run"] = k
                res.append(r)
                print(f"{name:18s} {MODE_NAMES[mode]:6s} run {k}: {r['ms_per_round']:8.3f} ms/round  {r['photons_per_s'] / 1e6:8.1f} M photons/s"
                      f"  deposit {r['deposit_ms']:7.3f} ms  ({time.time() - t0:.1f} s)", flush=True)
        _, _, P = config(name)
        out["workloads"][name] = dict(photons_per_round=P, warmup=warmup, steps=steps, results=res, summary={
            MODE_NAMES[m]: dict(photons_per_s=[x["photons_per_s"] for x in res if x["mode"] == m],
                                deposit_ms=[x["deposit_ms"] for x in res if x["mode"] == m]) for m in MODES})
    return out


def weak_scaling(args):
    import torch
    import torch.distributed as dist

    from cgraytracing_b200 import Context
    from cgraytracing_b200.binding import comm_destroy
    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer, make_native_comm

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    name = "c3_dragon_glass"
    scene, cfg, P = config(name)
    warmup, steps = STEPS[name]
    res = []
    for k in range(args.runs):
        for mode in (1, 2):
            comm = make_native_comm(local, rank, world)
            with Context(local) as g:
                g.set_config(cfg, accum_mode=mode)
                scene.build_into(g)
                g.commit()
                R = ShardedRenderer(GpuEngine(g, local, comm, world, rank=rank), rank, world)
                R.eye(cfg.height)
                for _ in range(warmup):
                    R.round(world * P)
                g.synchronize()
                dist.barrier()
                t0 = time.perf_counter()
                for _ in range(steps):
                    R.round(world * P)
                g.synchronize()
                dist.barrier()
                s = time.perf_counter() - t0
            comm_destroy(comm)  # after the context that used it
            res.append(dict(mode=mode, run=k, ms_per_round=1e3 * s / steps, photons_per_s=world * P * steps / s))
            if rank == 0:
                print(f"{world} GPUs {MODE_NAMES[mode]:6s} run {k}: {1e3 * s / steps:8.3f} ms/round", flush=True)
    out = dict(tool="tools/accum_bench.py", world=world, card=card(local), workload=name, photons_per_gpu_per_round=P, results=res)
    dist.destroy_process_group()
    return out if rank == 0 else None


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--workloads", nargs="+", default=list(bench.WORKLOADS), choices=list(bench.WORKLOADS))
    args = ap.parse_args()
    out = weak_scaling(args) if int(os.environ.get("WORLD_SIZE", "1")) > 1 else single_gpu(args)
    if out is not None:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
