"""SPPM against PPM on one BASELINE config: one JSON line with both estimators' rounds side by side.

  python tools/sppm_bench.py --config c3 [--rounds K] [--warmup W] [--photons P] [--mode jitter|corner]

For each estimator: device time per round (CUDA events on the library's stream around K rounds, profiling off) and photons/s; then K more
rounds with profiling on, and the per-round milliseconds of each phase from cgrt_get_timings (eye, grid, photon pass = trace + deposit
sort + deposit, update / fold). SPPM also reports its visible points per round. c4 compares SPPM with one sample per pixel per round
against PPM with the config's four. Writes nothing into the tree.
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=sorted(CONFIGS), default="c3")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--photons", type=int, default=0, help="photons per round (default: the config's 16 Mi)")
    ap.add_argument("--mode", choices=["jitter", "corner"], default="jitter")
    a = ap.parse_args()
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
