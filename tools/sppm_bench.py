"""SPPM against PPM on one BASELINE config: one JSON line with both estimators' rounds side by side.

  python tools/sppm_bench.py --config c3 [--rounds K] [--warmup W] [--photons P] [--mode jitter|corner]

For each estimator: device time per round (CUDA events on the library's stream around K rounds, profiling off) and photons/s; then K more
rounds with profiling on, and the per-round milliseconds of each phase from cgrt_get_timings (eye, grid, photon pass = trace + deposit
sort + deposit, update / fold). SPPM also reports its visible points per round. c4 compares SPPM with one sample per pixel per round
against PPM with the config's four. Writes nothing into the tree.

  python tools/sppm_bench.py --config c3 --gpus N [--baseline LINE.json]

Several GPUs of one box, weak scaling: N processes (torch.distributed.run, the library's own NCCL communicator), sharded PPM and sharded
SPPM side by side at the config's photons per GPU per round, float accumulators, the config's SPPM samples for both. Per estimator: device
time per round (the slowest rank), total photons/s, efficiency against the 1-GPU line given with --baseline (its ms per round over this
one's), and with profiling on, in a separate pass, the per-round milliseconds of the eye pass, the record all-gather, the grid build, the
photon pass and the all-reduce plus fold (update).
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CONFIGS = {  # preset, width, height, photons/round, dof, PPM samples, SPPM samples (bench.py's c3 and c4)
    "c3": ("c3_dragon_glass", 1024, 1024, 16 << 20, 0, 1, 1),
    "c4": ("c4_bump_dof", 1920, 1080, 16 << 20, 1, 4, 1),
}


def gpu_info():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], text=True).strip()
        name, power = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the line still says what was measured
        return {"gpu": "unknown (%s)" % type(e).__name__}


def run(mode, preset_name, cfg, photons, warmup, rounds):
    import torch

    from cgraytracing_b200 import Context, preset

    s = preset(preset_name)
    g = Context(0)
    g.set_config(cfg, accum_mode=1)
    s.build_into(g); g.commit()
    if mode:
        g.set_sppm(mode)
    else:
        g.eye_pass(); g.build_grid()
    r = 0
    visible = []

    def one_round():
        nonlocal r
        if mode:
            g.sppm_begin_round(r)
            visible.append(g.num_hitpoints())
        g.photon_pass(r * photons, photons)
        g.round_update()
        r += 1

    for _ in range(warmup):
        one_round()
    g.synchronize()
    stream = torch.cuda.ExternalStream(g.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(rounds):
        one_round()
    g.accum_dev()  # PPM's update runs on the library's side stream: make the timed stream wait for it
    e1.record(stream)
    g.synchronize()
    ms = e0.elapsed_time(e1) / rounds
    g.set_profiling(True)
    t0 = g.timings()
    for _ in range(rounds):
        one_round()
    g.synchronize()
    t1 = g.timings()
    d = {k: (t1[k] - t0[k]) / rounds for k in t0}
    out = {"ms_per_round": round(ms, 3), "photons_per_s": photons / (ms * 1e-3),
           "phase_ms_per_round_profiled": {"eye": round(d["eye"], 3), "grid": round(d["grid"], 3),
                                           "photon_pass": round(d["photon_trace"] + d["deposit_sort"] + d["photon_deposit"], 3),
                                           "photon_trace": round(d["photon_trace"], 3), "photon_deposit": round(d["photon_deposit"], 3),
                                           "update": round(d["update"], 3)},
           "hitpoints": g.num_hitpoints()}
    if mode:
        out["visible_points_per_round"] = {"mean": float(sum(visible) / len(visible)), "min": min(visible), "max": max(visible)}
        del out["hitpoints"]
    g.close()
    return out


def run_sharded(mode, preset_name, cfg, photons_per_gpu, warmup, rounds, rank, world, local, comm):
    import torch

    from cgraytracing_b200 import Context, preset
    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer

    s = preset(preset_name)
    g = Context(local)
    g.set_config(cfg, accum_mode=1)
    s.build_into(g); g.commit()
    R = ShardedRenderer(GpuEngine(g, local, comm, world, rank=rank, sppm=mode), rank, world)
    P = photons_per_gpu * world
    visible = []
    if not mode:
        R.eye(cfg.height)

    def one_round():
        if mode:
            R.eye(cfg.height)
            visible.append(g.num_hitpoints())
        R.round(P)

    for _ in range(warmup):
        one_round()
    g.synchronize()
    stream = torch.cuda.ExternalStream(g.stream(), device=torch.device("cuda", local))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(rounds):
        one_round()
    g.accum_dev()
    e1.record(stream)
    g.synchronize()
    ms = e0.elapsed_time(e1) / rounds
    g.set_profiling(True)
    t0 = g.timings()
    for _ in range(rounds):
        one_round()
    g.synchronize()
    t1 = g.timings()
    d = {k: (t1[k] - t0[k]) / rounds for k in t0}
    out = {"ms_per_round": ms,
           "phase_ms_per_round_profiled": {"eye": round(d["eye"], 3), "allgather": round(d["allgather"], 3), "grid": round(d["grid"], 3),
                                           "photon_pass": round(d["photon_trace"] + d["deposit_sort"] + d["photon_deposit"], 3),
                                           "update": round(d["update"], 3)},
           "hitpoints": g.num_hitpoints()}
    if mode:
        out["visible_points_per_round"] = {"mean": float(sum(visible) / len(visible)), "min": min(visible), "max": max(visible)}
        del out["hitpoints"]
    if comm is not None:
        g.set_comm(0, 1)
    g.close()
    return out


def sharded_main(a):
    """One rank of `--gpus N` (under torch.distributed.run)."""
    import torch
    import torch.distributed as dist

    from cgraytracing_b200 import RenderConfig
    from cgraytracing_b200.binding import comm_destroy
    from cgraytracing_b200.distributed import make_native_comm

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    name, W, H, P, dof, ppm_spp, sppm_spp = CONFIGS[a.config]
    P = a.photons or P
    mode = {"jitter": 1, "corner": 2}[a.mode]
    comm = make_native_comm(local, rank, world) if world > 1 else None
    cfg = RenderConfig(width=W, height=H, use_dof=dof, num_of_samples=sppm_spp)
    res = {}
    for key, m in (("ppm", 0), ("sppm", mode)):
        mine = run_sharded(m, name, cfg, P, a.warmup, a.rounds, rank, world, local, comm)
        every = [None] * world
        dist.all_gather_object(every, mine)
        mine["ms_per_round"] = max(e["ms_per_round"] for e in every)  # a round ends when the slowest rank's does
        mine["ms_per_round_min_rank"] = round(min(e["ms_per_round"] for e in every), 3)
        mine["ms_per_round"] = round(mine["ms_per_round"], 3)
        mine["photons_per_s"] = P * world / (mine["ms_per_round"] * 1e-3)
        res[key] = mine
    if comm is not None:
        comm_destroy(comm)
    if rank == 0:
        base = json.load(open(a.baseline)) if a.baseline else None
        for key in ("ppm", "sppm"):
            res[key]["efficiency_vs_1gpu"] = round(base[key]["ms_per_round"] / res[key]["ms_per_round"], 3) if base else None
        line = {"tool": "sppm_bench", "gpus": world, "scaling": "weak", "config": a.config, "preset": name, "width": W, "height": H,
                "photons_per_round_per_gpu": P, "rounds": a.rounds, "warmup": a.warmup, "accum_mode": 1, "sppm_mode": a.mode, "samples": sppm_spp,
                "collectives": "native NCCL communicator" if world > 1 else "none", "ppm": res["ppm"], "sppm": res["sppm"],
                "sppm_round_over_ppm_round": round(res["sppm"]["ms_per_round"] / res["ppm"]["ms_per_round"], 3)}
        line.update(gpu_info())
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c3")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--photons", type=int, default=0, help="photons per round (default: the config's 16 Mi)")
    ap.add_argument("--mode", choices=["jitter", "corner"], default="jitter")
    ap.add_argument("--gpus", type=int, default=0, help="N >= 1: sharded PPM and SPPM over N GPUs of this box, N processes (weak scaling)")
    ap.add_argument("--baseline", default="", help="with --gpus: the --gpus 1 line of the same config, for the efficiency")
    a = ap.parse_args()
    if a.gpus:
        if "RANK" in os.environ:
            return sharded_main(a)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(a.gpus), "--master-addr", "127.0.0.1",
               "--master-port", "29541", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    from cgraytracing_b200 import RenderConfig

    name, W, H, P, dof, ppm_spp, sppm_spp = CONFIGS[a.config]
    P = a.photons or P
    mode = {"jitter": 1, "corner": 2}[a.mode]
    ppm = run(0, name, RenderConfig(width=W, height=H, use_dof=dof, num_of_samples=ppm_spp), P, a.warmup, a.rounds)
    sppm = run(mode, name, RenderConfig(width=W, height=H, use_dof=dof, num_of_samples=sppm_spp), P, a.warmup, a.rounds)
    line = {"tool": "sppm_bench", "config": a.config, "preset": name, "width": W, "height": H, "photons_per_round": P, "rounds": a.rounds,
            "warmup": a.warmup, "accum_mode": 1, "sppm_mode": a.mode, "ppm_samples": ppm_spp, "sppm_samples": sppm_spp,
            "ppm": ppm, "sppm": sppm, "sppm_round_over_ppm_round": round(sppm["ms_per_round"] / ppm["ms_per_round"], 3)}
    line.update(gpu_info())
    print(json.dumps(line))


if __name__ == "__main__":
    main()
