#!/usr/bin/env python
"""bench.py — photons/s of the B200 photon-mapping hot path on the configuration the north star names:
the glass dragon (100,000 triangles) + chessboard floor at 1024x1024, one round = 16 Mi photons per GPU
(BASELINE.json configs[2], "c3_dragon_glass": 50 rounds x 16M photons).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A *step* is one round of the hot path: trace `--photons` photons per GPU against the persistent hitpoint set (emission,
closest hit, bounces, 27-cell deposits), all-reduce the per-hitpoint accumulators when N > 1, per-round radius/flux update.
`value` times K rounds on the device (inputs resident: scene, BVH, hitpoints, grid). `--dump-outputs DIR` writes the hitpoint
state the last timed round left (see dump_outputs), so that two builds can be compared output for output. `e2e` times the whole render()
of the named config through the C ABI from HOST buffers: scene H2D + LBVH build + eye pass + grid + `--e2e-rounds` rounds +
image D2H, wall clock. `roofline` comes from a separate profiled round of the same run (every kernel launch bracketed by
CUDA events on the library's stream). Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# BASELINE.json configs. The headline (default) is c3: it is the config the metric is quoted on and it fits one GPU.
WORKLOADS = {
    #  name                preset               width height photons/round rounds hashsize  dof samples
    "c1_spheres_bezier": ("c1_spheres_bezier", 512, 512, 1 << 20, 10, 1000001, 0, 1),
    "c2_bunny_chess": ("c2_bunny_chess", 1024, 1024, 4 << 20, 20, 1000001, 0, 1),
    "c3_dragon_glass": ("c3_dragon_glass", 1024, 1024, 16 << 20, 50, 1000001, 0, 1),
    "c4_bump_dof": ("c4_bump_dof", 1920, 1080, 16 << 20, 20, 1000001, 1, 4),
    "c5_dragon_4096": ("c3_dragon_glass", 4096, 4096, 1 << 30, 1, 16777259, 0, 1),  # 1 Gi photons per round; hashsize raised (SURVEY 7.6)
}
WORKLOAD = "c3_dragon_glass"
PRESET, WIDTH, HEIGHT, PHOTONS_PER_ROUND, ROUNDS, HASHSIZE, USE_DOF, SAMPLES = WORKLOADS[WORKLOAD]


def select_workload(name):
    global WORKLOAD, PRESET, WIDTH, HEIGHT, PHOTONS_PER_ROUND, ROUNDS, HASHSIZE, USE_DOF, SAMPLES
    WORKLOAD = name
    PRESET, WIDTH, HEIGHT, PHOTONS_PER_ROUND, ROUNDS, HASHSIZE, USE_DOF, SAMPLES = WORKLOADS[name]


def make_config(RenderConfig, **kw):
    return RenderConfig(width=WIDTH, height=HEIGHT, hashsize=HASHSIZE, use_dof=USE_DOF, num_of_samples=SAMPLES, **kw)

# SURVEY.md section 8(d): algorithmic bytes per unit (layout-independent record sizes)
B_SEGMENT, B_NODE, B_TRI = 80, 32, 48
B_CELLS, B_CAND, B_DEP = 27 * 8, 32, 32


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def deposit_record_bytes(ctx):
    from cgraytracing_b200.binding import load_library

    return int(load_library().cgrt_deposit_record_bytes(ctx.h))


def load_ncu_traffic(photons, accum):
    """DRAM bytes per round (dram__bytes_read.sum + dram__bytes_write.sum summed over the round's launches of each kernel family) from
    the committed ncu pass of this command line, if one matches the configuration: profiles/ncu_traffic.json, written by
    tools/make_ncu_traffic.py from the launch list it names."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        t = json.load(f)
    c = t.get("config", {})
    if c.get("workload") != WORKLOAD or c.get("photons") != photons or c.get("accum") != accum:
        return None
    out = dict(t["bytes_per_round"])
    out["source"] = t.get("source")
    return out


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU arms (the only places bench.py touches oracle/)
# ---------------------------------------------------------------------------------------------------------------------
def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def host_threads():
    """CPUs this process may run on. NOT omp_get_max_threads(): torchrun exports OMP_NUM_THREADS=1 to its workers."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def shrink_radii_like_gpu_rounds(o, rounds):
    """Put the oracle's hitpoints where the GPU's are when its timed rounds start: after `rounds` updates with the same number M of
    accepted photons per round every hitpoint has r2 = r0^2 * prod_k k*a / ((k-1)*a + 1) (the U2 rule with equal M, whatever M is), so
    the same updates are applied here with an artificial M instead of tracing 16 Mi photons per warm-up round on the CPU."""
    n = o.num_hitpoints()
    for _ in range(rounds):
        o.upload_accum(np.zeros((n, 3)), np.full(n, 1000.0))
        o.round_update()


def as_shipped_leg(scene, photons_per_thread, threads):
    """The UNMODIFIED reference (oracle/_ref/libcgref.so = /root/reference/main.cpp + headers compiled in place): its own trace(),
    Hashtable, glibc rand() under its global lock and the nested `omp parallel for` of main.cpp:222-249, at its compiled-in image size."""
    from oracle import binding as ob

    if not ob.have_ref():
        return None
    r = ob.Ref(scene)
    w, h = r.image_size()
    t0 = time.time()
    r.eye_pass_as_shipped()
    t_eye = time.time() - t0
    sec = r.photon_loop_as_shipped(photons_per_thread, threads, seed=1)
    total = photons_per_thread * threads
    return {"value": total / sec, "unit": "photons/s", "cores": threads, "kind": "reference", "seconds": sec, "eye_pass_seconds": t_eye,
            "image": [w, h], "hitpoints": r.num_hitpoints(),
            "sample": f"main.cpp:222-249 as shipped: {threads} threads x {photons_per_thread} photons each (every thread runs the whole loop), "
                      f"rand() lock included, U1 per-photon update, compiled-in {w}x{h} image of the same scene"}


def cpu_baseline(scene, cfg, photons, threads=None, warm_rounds=0, shipped_photons=0):
    """The CPU oracle (a line-by-line port of the reference, thread-local Philox, U2 accumulators) on the host cores."""
    from oracle import binding as ob

    o = ob.Oracle(scene, cfg)
    threads = threads or host_threads()
    t0 = time.time()
    o.eye_pass()
    t_eye = time.time() - t0
    shrink_radii_like_gpu_rounds(o, warm_rounds)
    c0 = o.counters()
    sec = o.photon_pass(warm_rounds * PHOTONS_PER_ROUND, photons, threads)
    c = o.counters()
    hits = max(1, c["diffuse_hits"] - c0["diffuse_hits"])
    out = {
        "value": photons / sec, "unit": "photons/s", "cores": threads, "kind": "port", "cpu_model": cpu_model(),
        "sample": f"{photons} photons of the same scene/config on {threads} OpenMP threads after a full single-thread eye pass, radii as "
                  f"after {warm_rounds} rounds (where the GPU's timed rounds start)",
        "eye_rays_per_s": c["eye_segments"] / t_eye, "eye_threads": 1, "seconds": sec,
        "deposits_per_hit": (c["deposits"] - c0["deposits"]) / hits, "candidates_per_hit": (c["candidates"] - c0["candidates"]) / hits,
        "node_visits_per_segment": c["node_visits"] / max(1, c["eye_segments"] + c["photon_segments"]),
    }
    if shipped_photons > 0:
        out["as_shipped"] = as_shipped_leg(scene, max(1, shipped_photons // threads), threads)
    return out


DUMP_BYTES = 64_000_000  # all files of --dump-outputs together
NPY_HEADER = 128
DUMP_NAMES = ("hitpoint_flux", "hitpoint_r2", "hitpoint_n", "hitpoint_index")


def dump_outputs(out_dir, hp, limit=DUMP_BYTES):
    """Writes what a round leaves for its caller, the per-hitpoint state in canonical order, as float64 .npy files: hitpoint_flux
    [n, 3], hitpoint_r2 [n], hitpoint_n [n] (accepted-photon counts). When that exceeds `limit` bytes, the same seeded sample of
    rows is taken from each array and the sampled row numbers go to hitpoint_index.npy. Files of an earlier dump into the same
    directory are removed first, so that a stale hitpoint_index.npy never sits beside whole arrays."""
    arrays = {"hitpoint_flux": hp["flux"], "hitpoint_r2": hp["r2"], "hitpoint_n": hp["n"]}
    n = len(hp["r2"])
    row_bytes = 8 * sum(a[:1].size for a in arrays.values())
    if n * row_bytes + len(arrays) * NPY_HEADER > limit:
        k = (limit - (len(arrays) + 1) * NPY_HEADER) // (row_bytes + 8)
        rows = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["hitpoint_index"] = rows
    os.makedirs(out_dir, exist_ok=True)
    for name in DUMP_NAMES:
        path = os.path.join(out_dir, name + ".npy")
        if os.path.exists(path):
            os.remove(path)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_reference(args):
    """The reference arm: the CPU implementation of the path on ALL host cores of the box. The timed value is the oracle port (pinned bit
    for bit to the compiled reference, lock-free Philox streams: the STRONGER baseline); the unmodified reference binary's own loop, which
    spends most of its time in glibc's rand() lock, is timed beside it (`cpu_baseline.as_shipped`)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from cgraytracing_b200.scene import RenderConfig, preset
    from oracle import binding as ob

    scene = preset(PRESET)
    cfg = make_config(RenderConfig, update_mode=1, into_rule=0)
    o = ob.Oracle(scene, cfg)
    threads = host_threads()
    o.eye_pass(nthreads=threads)
    shrink_radii_like_gpu_rounds(o, max(0, 3 - args.warmup))  # the GPU arm's timed rounds start after >= 3 rounds
    sample = args.ref_photons
    times = []
    c0 = None
    for s in range(args.warmup + args.steps):
        if s == args.warmup:
            c0 = o.counters()
        sec = o.photon_pass(s * sample, sample, threads)
        o.round_update()
        if s >= args.warmup:
            times.append(sec)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o.download_hitpoints(fields=("flux", "r2", "n")))
    c1 = o.counters()
    total = sum(times)
    v = sample * len(times) / total
    hits = max(1, c1["diffuse_hits"] - c0["diffuse_hits"])
    shipped = as_shipped_leg(scene, max(1, args.shipped_photons // threads), threads) if args.shipped_photons > 0 else None
    line = {
        "impl": "reference", "metric": "photons_per_s", "value": v, "unit": "photons/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "width": WIDTH, "height": HEIGHT, "photons_per_step": sample,
                   "note": "bounded CPU sample of the same round; cost per photon is stationary"},
        "cpu_baseline": {"value": v, "unit": "photons/s", "cores": threads, "kind": "port", "cpu_model": cpu_model(),
                         "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS"),
                         "deposits_per_hit": (c1["deposits"] - c0["deposits"]) / hits,
                         "sample": f"{sample} photons per step x {args.steps} steps, oracle port of main.cpp trace()/render() "
                                   f"(pinned bit-exact to the compiled reference), {threads} OpenMP threads",
                         "as_shipped": shipped},
        "e2e": {"value": v, "unit": "photons/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit_line(line)


# ---------------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    from cgraytracing_b200 import Context, RenderConfig, preset
    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer, make_native_comm, row_shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    scene = preset(PRESET)
    cfg = make_config(RenderConfig)
    # c5 is defined as 1 Gi photons per round IN TOTAL (the scaling sweep of the north star): strong scaling, every other workload
    # keeps the photons per GPU fixed (weak scaling)
    strong = WORKLOAD == "c5_dragon_4096" and args.photons <= 0
    P = args.photons if args.photons > 0 else (PHOTONS_PER_ROUND // world if strong else PHOTONS_PER_ROUND)
    peak, peak_src = load_peaks()

    # ---- setup (untimed for `value`): scene upload + LBVH build, tile-sharded eye pass + all-gather, grid
    # a throw-away context first: it pays the process's one-time costs (module load, cudaMalloc of the arena blocks, which the
    # library keeps for the process), so that the timed setup below is what every later render() in this process pays
    with Context(local) as gw:
        gw.set_config(cfg, accum_mode=args.accum)
        scene.build_into(gw); gw.commit()
        y0w, y1w = row_shard(HEIGHT, rank, world)
        gw.eye_pass(y0w, y1w); gw.build_grid()
        tmw = gw.timings()
    g = Context(local)
    g.set_config(cfg, accum_mode=args.accum)
    g.set_overlap(bool(args.overlap))
    scene.build_into(g)
    t0 = time.time()
    g.commit()
    t_commit = time.time() - t0
    # N > 1: both collectives of the path (all-gather of the eye tiles' hitpoint records, all-reduce of the accumulators) run inside the
    # library over its own NCCL communicator; --collective torch leaves the all-reduce to torch.distributed on the library's stream
    comm = make_native_comm(local, rank, world) if (world > 1 and args.collective in ("native", "peer")) else None
    peer = args.collective == "peer"
    eng = GpuEngine(g, local, comm, world, rank=rank, peer=peer)
    R = ShardedRenderer(eng, rank, world)
    R.eye(HEIGHT)
    g.synchronize()
    tm0 = g.timings()
    c0 = g.counters()

    # ---- roofline accounting (outside the timed region): counting build of the same traversal on a sample
    per_seg_nodes = per_seg_tris = None
    eye_warm = (c0["eye_segments"], tm0["eye"], tm0["grid"])  # this rank's tile of the image (the whole image at world 1)
    if rank == 0:
        with Context(local) as gc:
            gc.set_config(cfg, accum_mode=args.accum)
            scene.build_into(gc); gc.commit(); gc.eye_pass(); gc.build_grid()
            gc.set_counting(True)
            gc.photon_pass(0, min(P, 1 << 20))
            cc = gc.counters()
            per_seg_nodes = cc["node_visits"] / cc["photon_segments"]
            per_seg_tris = cc["tri_tests"] / cc["photon_segments"]

    for _ in range(args.warmup):
        R.round(world * P)
    g.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    c1 = g.counters()
    stream = torch.cuda.ExternalStream(g.stream())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        R.round(world * P)
    g.accum_dev()  # the last round's all-reduce + update run on the library's side stream: make the timed stream wait for them
    e1.record(stream)
    g.synchronize()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.result()
    ms = e0.elapsed_time(e1)
    c2 = g.counters()
    if args.dump_outputs and rank == 0:  # every rank holds the same state after a round's update
        dump_outputs(args.dump_outputs, g.download_hitpoints(fields=("flux", "r2", "n")))
    if world > 1:
        t = torch.tensor([ms], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    total_photons = world * P * args.steps
    value = total_photons / (ms * 1e-3)

    # ---- one profiled round (every launch bracketed by events on the ctx stream): per-kernel durations for the roofline
    g.set_profiling(True)
    tp0, cp0 = g.timings(), g.counters()
    R.round(world * P)
    g.synchronize()
    tp1, cp1 = g.timings(), g.counters()
    g.set_profiling(False)

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # eye pass of the whole image: segments of all tiles / the slowest tile's device time (pass + grid are per rank)
    eye_segments_all = sum_over_ranks(c0["eye_segments"])
    eye_ms_all = max_over_ranks(tm0["eye"])

    # ---- the same K rounds with fp64 accumulators (bit-exact deposits; the headline runs float accumulators), one GPU only
    value_f64 = None
    if args.accum == 1 and world == 1 and args.f64_too:
        with Context(local) as g0:
            g0.set_config(cfg, accum_mode=0)
            scene.build_into(g0); g0.commit(); g0.eye_pass(); g0.build_grid()
            for k in range(args.warmup):
                g0.photon_pass(k * P, P); g0.round_update()
            g0.synchronize()
            s0 = torch.cuda.ExternalStream(g0.stream())
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(s0)
            for k in range(args.steps):
                g0.photon_pass((args.warmup + k) * P, P); g0.round_update()
            g0.accum_dev()
            f1.record(s0)
            g0.synchronize()
            value_f64 = P * args.steps / (f0.elapsed_time(f1) * 1e-3)

    # ---- e2e: the whole render() of the named config through the C ABI from HOST buffers, on all N GPUs (tile-sharded eye pass,
    # all-gather of the hitpoint records, photon shards, all-reduce per round, image download), wall clock, max over ranks
    scene_bytes = sum(o["tri9"].nbytes for o in scene.objects if o["kind"] == "mesh") + sum(t["rgb"].nbytes for t in scene.textures)
    e2e = None
    if args.e2e_rounds > 0:
        def render_once(rounds):
            if world > 1:
                dist.barrier()
            t0 = time.time()
            with Context(local) as ge:
                ge.set_config(cfg, accum_mode=args.accum)
                scene.build_into(ge); ge.commit()
                Re = ShardedRenderer(GpuEngine(ge, local, comm, world, rank=rank, peer=peer), rank, world)
                Re.eye(HEIGHT)
                for _ in range(rounds):
                    Re.round(world * P)
                img, rgb8 = ge.gather_image(float(Re.emitted), want_rgb8=True)
            return max_over_ranks(time.time() - t0), img, rgb8

        render_once(1)  # warm-up (memory pool, module load)
        t1, img, rgb8 = render_once(1)
        tN, img, rgb8 = render_once(args.e2e_rounds)
        e2e = {"value": world * P * args.e2e_rounds / tN, "unit": "photons/s", "h2d_bytes_per_step": int(scene_bytes),
               "d2h_bytes_per_step": int(img.nbytes + rgb8.nbytes), "seconds_per_step": tN, "rounds_per_step": args.e2e_rounds,
               "one_round_render": {"value": world * P / t1, "seconds": t1},
               "what": f"one step = one whole render() of {WORKLOAD} on {world} GPU(s): cgrt_create + scene upload from host arrays + LBVH build + "
                       f"eye pass (image rows sharded over the ranks, hitpoint records all-gathered) + grid + {args.e2e_rounds} rounds x "
                       f"{world * P} photons + all-reduce + updates + fp64 image and 8-bit image download on every rank, wall clock, max over ranks"}

    photon_chunk = g.photon_chunk()
    rec_b = deposit_record_bytes(g)
    g.close()  # every rank at the same point: with the peer exchange a context's shutdown is a handshake between the ranks
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    seg = cp1["photon_segments"] - cp0["photon_segments"]
    hits = cp1["diffuse_hits"] - cp0["diffuse_hits"]
    gathered = cp1["gathered_hits"] - cp0["gathered_hits"]  # hits that went through the 27-cell gather (the rest were culled)
    cand = cp1["candidates"] - cp0["candidates"]
    dep = cp1["deposits"] - cp0["deposits"]
    groups = cp1["cell_groups"] - cp0["cell_groups"]
    staged = cp1["staged_candidates"] - cp0["staged_candidates"]
    dt = lambda k: (tp1[k] - tp0[k]) * 1e-3
    t_trace, t_dep, t_upd, t_sort = dt("photon_trace"), dt("photon_deposit"), dt("update"), dt("deposit_sort")
    t_emit, t_trav, t_cont = dt("trace_emit"), dt("trace_traverse"), dt("trace_continue")
    n_chunks = (P + photon_chunk - 1) // max(1, photon_chunk)
    # (1) SURVEY 8(d): bytes the REFERENCE's algorithm touches for the same work, in device-layout record sizes
    bytes_trace = seg * (B_SEGMENT + B_NODE * per_seg_nodes + B_TRI * per_seg_tris)
    bytes_dep_survey = gathered * B_CELLS + cand * B_CAND + dep * B_DEP
    # (2) compulsory bytes of THIS deposit kernel: every sorted record and its order entry once, the 27 bucket ranges and every
    # bucket entry's filter records once per cell GROUP (the hits of a group share them in shared memory), one accumulator update per deposit
    cand_b = 48 if args.accum == 1 else 32
    acc_b = 16 if args.accum == 1 else 32 + 32
    bytes_dep = gathered * (rec_b + 4) + groups * B_CELLS + staged * cand_b + dep * acc_b
    # the trace family also writes the deposit table (record + bin per recorded hit) and the counting sort reads the bins and writes the order
    bytes_table_write = gathered * (rec_b + 4)
    bytes_sort = P * cfg.max_depth * 4 + gathered * 4
    traffic = load_ncu_traffic(P, args.accum)
    t_all = t_trace + t_dep + t_sort + t_upd
    kernels = {
        "photon_trace_family": {"seconds": t_trace, "alg_bytes": bytes_trace, "gbps": bytes_trace / t_trace / 1e9, "launches": 11 * n_chunks,
                                "ms_per_round": 1e3 * t_trace, "nodes_per_segment": per_seg_nodes, "tris_per_segment": per_seg_tris,
                                "segments_per_s": seg / t_trace, "deposit_table_write_bytes": bytes_table_write,
                                "split_ms": {"photon_trace_kernel<emission> x1": 1e3 * t_emit, "photon_traverse_kernel x5": 1e3 * t_trav,
                                             "photon_trace_kernel<continuation> x5": 1e3 * t_cont}},
        "photon_deposit_kernel": {"seconds": t_dep, "alg_bytes": bytes_dep, "gbps": bytes_dep / t_dep / 1e9, "launches": n_chunks,
                                  "ms_per_launch": 1e3 * t_dep / n_chunks, "candidates_per_hit": cand / max(1, hits),
                                  "deposits_per_hit": dep / max(1, hits), "hits_per_s": hits / t_dep, "diffuse_hits": hits, "gathered_hits": gathered,
                                  "cell_groups": groups, "staged_candidates": staged, "hits_per_group": gathered / max(1, groups),
                                  "exact_tests_per_hit": (cp1["exact_tests"] - cp0["exact_tests"]) / max(1, hits),
                                  "reference_algorithm_bytes": bytes_dep_survey,
                                  "reference_algorithm_gbps": bytes_dep_survey / t_dep / 1e9},
        "bin_scan+bin_scatter_kernel": {"seconds": t_sort, "alg_bytes": bytes_sort, "gbps": bytes_sort / max(t_sort, 1e-9) / 1e9, "launches": 3 * n_chunks},
        "round_update_kernel": {"seconds": t_upd, "launches": 1},
    }
    # the roofline entry is the kernel family with the largest share of the step
    dom = max(("photon_trace_family", "photon_deposit_kernel"), key=lambda k: kernels[k]["seconds"])
    sum_bytes = bytes_trace + bytes_table_write + bytes_dep + bytes_sort
    def entry(k):
        v = kernels[k]
        tr = traffic.get(k) if traffic else None
        return {"achieved": v["gbps"], "frac": v["gbps"] / peak, "share_of_step": v["seconds"] / t_all, "traffic": tr,
                "dram_frac": (tr / v["seconds"] / 1e9 / peak) if tr else None}
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["gbps"], "peak": peak, "unit": "GB/s", "frac": kernels[dom]["gbps"] / peak,
                "traffic": entry(dom)["traffic"], "peak_source": peak_src, "share_of_step": kernels[dom]["seconds"] / t_all,
                "dram_frac": entry(dom)["dram_frac"], "traffic_source": traffic.get("source") if traffic else None,
                "other_kernel": {k: entry(k) for k in kernels if k != dom and "gbps" in kernels[k]},
                "whole_step": {"alg_bytes": sum_bytes, "gbps": sum_bytes / t_all / 1e9, "frac": sum_bytes / t_all / 1e9 / peak},
                "note": "achieved = algorithmic bytes of the profiled round / CUDA-event duration of the launches. Trace family: SURVEY 8(d), 80 B per segment + "
                        "32 B per node visit + 48 B per triangle test (counting build of the same traversal). Deposit kernel: the compulsory bytes of "
                        "its own design — sorted record + order entry per gathered hit, 27 x 8 B of bucket ranges and the bucket entries' filter "
                        "records once per CELL GROUP (hits of one cell share them in shared memory), one accumulator update per deposit; the reference "
                        "algorithm's per-hit figure (27*8 + 32 per scanned candidate + 32 per deposit) is reported beside it as "
                        "reference_algorithm_gbps and is not a bound. No kernel of this path is HBM-bound: the trace family is bound by divergence and "
                        "dependent L2 latency, the deposit kernel by the shared-memory pipe (profiles/). whole_step = all algorithmic bytes of a round "
                        "over the round's device time. traffic = DRAM bytes per round from the committed ncu pass named in traffic_source (null when "
                        "no capture of this configuration is committed). peak = measured HBM copy bandwidth"}

    # ---- CPU baseline beside it (bounded sample)
    cpu = cpu_baseline(scene, make_config(RenderConfig, update_mode=1, into_rule=0), args.cpu_photons, warm_rounds=args.warmup,
                       shipped_photons=args.shipped_photons) if (args.cpu_photons > 0 and world == 1) else None

    line = {
        "metric": "photons_per_s", "value": value, "unit": "photons/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f64 decisions / f64 accumulators" if args.accum == 0 else "f64 decisions / f32 accumulators",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "width": WIDTH, "height": HEIGHT, "photons_per_gpu_per_step": P, "hitpoints": c2["hitpoints"],
                   "triangles": scene.num_triangles(), "accum": "f64 atomics" if args.accum == 0 else "v4.f32 red",
                   "collective": (args.collective if world > 1 else None),
                   "l2": f"inputs larger than L2: every round writes and re-reads a fresh deposit table ({P} photons x {cfg.max_depth} bounces x "
                         f"{rec_b} B slots) and new photons"},
        "value_f64_accumulators": value_f64,
        "s_per_round": ms * 1e-3 / args.steps, "eye_rays_per_s": eye_segments_all / (eye_ms_all * 1e-3),
        "segments_per_s": (c2["photon_segments"] - c1["photon_segments"]) * world / (ms * 1e-3),
        "setup": {"commit_s": t_commit, "eye_ms_first_context": tmw["eye"], "grid_ms_first_context": tmw["grid"], "eye_ms": eye_warm[1],
                  "grid_ms": eye_warm[2], "eye_segments": eye_warm[0],
                  "eye_segments_all_ranks": eye_segments_all, "eye_ms_slowest_rank": eye_ms_all,
                  "note": "eye_rays_per_s = segments of the whole image (all ranks' row tiles) / the slowest rank's eye-pass device time (all "
                          "bounce launches) in the second context of the process; the first context also pays the cudaMalloc of the arena "
                          "blocks the library then keeps"},
        "roofline": roofline, "kernels": kernels, "cpu_baseline": cpu, "clocks": clocks, "e2e": e2e,
        "gpu_launches": int(c2["gpu_launches"] - c1["gpu_launches"]),
    }
    emit_line(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=WORKLOAD, choices=sorted(WORKLOADS), help="BASELINE.json config (default: the headline config c3)")
    ap.add_argument("--photons", type=int, default=0, help="photons per GPU per step (default: the workload's photons per round; c3 = 16 Mi)")
    ap.add_argument("--accum", type=int, default=1, help="0: fp64 atomics, 1: one v4.f32 red per deposit (SURVEY 8e: float32 x4 accumulators)")
    ap.add_argument("--overlap", type=int, default=0, help="1: trace of round r+1 overlaps the deposit of round r on a second stream")
    ap.add_argument("--cpu-photons", type=int, default=400000, help="photon budget of the CPU baseline sample (0 = skip)")
    ap.add_argument("--ref-photons", type=int, default=200000, help="photons per step of --impl reference")
    ap.add_argument("--shipped-photons", type=int, default=100000, help="total photons of the 'reference as shipped' leg (oracle/_ref; 0 = skip)")
    ap.add_argument("--collective", default="native", choices=["native", "peer", "torch"],
                    help="N > 1: how the accumulators of a round are exchanged. native: ncclAllReduce inside the library, in stream order (fastest at "
                         "8 GPUs); peer: over peer memory inside the library, fused with the update and overlapped with the next round's trace (no "
                         "collective call in a round; fastest at 2 GPUs); torch: torch.distributed all-reduce on the library's stream")
    ap.add_argument("--f64-too", type=int, default=1, help="1: also time the same rounds with fp64 accumulators (value_f64_accumulators)")
    ap.add_argument("--e2e-rounds", type=int, default=-1, help="rounds of the end-to-end render() (default: the workload's own, c3 = 50; 0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the hitpoint state the last one left as DIR/<name>.npy "
                                                          "(float64, at most 64 MB in all; a seeded sample of the hitpoints beyond that)")
    args = ap.parse_args()
    select_workload(args.workload)
    if args.e2e_rounds < 0:
        args.e2e_rounds = ROUNDS
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


class _QuietStdout:
    """Everything native libraries print on fd 1 while the benchmark runs (NCCL's version banner, for one) goes to stderr, so that the
    JSON line is the only thing on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def emit(self, text):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(text, flush=True)
        os.dup2(2, 1)

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


_OUT = None


def emit_line(line):
    text = json.dumps(line)
    if _OUT is not None:
        _OUT.emit(text)
    else:
        print(text, flush=True)


if __name__ == "__main__":
    with _QuietStdout() as _OUT:
        main()
