"""bench.py's output contract, on the CPU-runnable arm (`--impl reference` times the oracle port on host cores)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_exactly_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-photons", "4000",
                        "--workload", "c2_bunny_chess"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["metric"] == "photons_per_s" and d["unit"] == "photons/s" and d["higher_is_better"] is True
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "c2_bunny_chess"
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0


def test_reference_arm_uses_every_host_core_under_torchrun_and_times_the_reference_as_shipped():
    """torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: the CPU arm must still use the cores the process may run on (affinity
    mask), and carry the unmodified reference's own photon loop (oracle/_ref, main.cpp:222-249) beside the port."""
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-photons", "4000",
                        "--shipped-photons", "2000", "--workload", "c2_bunny_chess"], capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    cb = d["cpu_baseline"]
    assert cb["cores"] == len(os.sched_getaffinity(0)) and cb["omp_num_threads_env"] == "1"
    assert cb["kind"] == "port" and cb["deposits_per_hit"] > 0
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libcgref.so")):
        sh = cb["as_shipped"]
        assert sh["kind"] == "reference" and sh["value"] > 0 and sh["cores"] == cb["cores"] and sh["hitpoints"] > 0


def _bench_with_dump(out, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
    files = sorted(out.iterdir())
    assert [f.name for f in files] == ["hitpoint_flux.npy", "hitpoint_n.npy", "hitpoint_r2.npy"]
    assert sum(f.stat().st_size for f in files) <= 64_000_000
    D = {f.stem: np.load(f) for f in files}
    assert all(a.dtype == np.float64 for a in D.values())
    return d, D


def test_reference_arm_dumps_the_state_its_last_step_left(oracle_lib, tmp_path):
    """The dump equals the same rounds replayed here through the oracle; same arguments, same inputs: the accepted-photon counts and
    the radii they set repeat exactly from run to run; one step fewer leaves fewer counts."""
    from cgraytracing_b200 import RenderConfig, preset

    P, W, S = 4000, 1, 2
    args = ("--impl", "reference", "--warmup", str(W), "--ref-photons", str(P), "--workload", "c2_bunny_chess", "--shipped-photons", "0")
    runs = [_bench_with_dump(tmp_path / f"run{i}", *args, "--steps", str(s)) for i, s in enumerate((S, S, S - 1))]
    (d, a), (_, b), (_, c) = runs
    assert d["steps"] == S and len(a["hitpoint_r2"]) == len(a["hitpoint_n"]) == len(a["hitpoint_flux"]) > 1000
    assert np.array_equal(a["hitpoint_n"], b["hitpoint_n"]) and np.array_equal(a["hitpoint_r2"], b["hitpoint_r2"])
    assert np.allclose(a["hitpoint_flux"], b["hitpoint_flux"], rtol=1e-9, atol=1e-12)
    assert a["hitpoint_n"].sum() > c["hitpoint_n"].sum() > 0
    # the reference arm: eye pass, radii as after the GPU arm's first 3 rounds (less the warm-up), then warm-up + timed rounds
    o = oracle_lib.Oracle(preset("c2_bunny_chess"), RenderConfig(width=1024, height=1024, hashsize=1000001, update_mode=1, into_rule=0))
    o.eye_pass(nthreads=o.max_threads())
    n = o.num_hitpoints()
    for _ in range(3 - W):
        o.upload_accum(np.zeros((n, 3)), np.full(n, 1000))
        o.round_update()
    for s in range(W + S):
        o.photon_pass(s * P, P, o.max_threads())
        o.round_update()
    hp = o.download_hitpoints(fields=("flux", "r2", "n"))
    assert np.array_equal(a["hitpoint_n"], hp["n"]) and np.array_equal(a["hitpoint_r2"], hp["r2"])
    assert np.allclose(a["hitpoint_flux"], hp["flux"], rtol=1e-9, atol=1e-12)


def test_dump_takes_the_same_seeded_rows_of_every_array_beyond_the_limit(tmp_path):
    import bench

    n = 5000
    hp = {"flux": np.arange(3.0 * n).reshape(n, 3), "r2": np.arange(n) + 0.5, "n": np.arange(n, dtype=np.int32)}
    for out in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(out), hp, limit=60000)
        assert sum(f.stat().st_size for f in out.iterdir()) <= 60000
    a, b = ({f.stem: np.load(f) for f in out.iterdir()} for out in (tmp_path / "a", tmp_path / "b"))
    rows = a["hitpoint_index"]
    assert 1000 < len(rows) < n and np.all(np.diff(rows) > 0) and all(v.dtype == np.float64 for v in a.values())
    assert np.array_equal(a["hitpoint_n"], rows) and np.array_equal(a["hitpoint_r2"], rows + 0.5) and np.array_equal(a["hitpoint_flux"][:, 0], 3 * rows)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # a whole dump into the same directory leaves no row numbers of the sampled one behind
    bench.dump_outputs(str(tmp_path / "a"), hp)
    assert sorted(f.name for f in (tmp_path / "a").iterdir()) == ["hitpoint_flux.npy", "hitpoint_n.npy", "hitpoint_r2.npy"]
    assert np.array_equal(np.load(tmp_path / "a" / "hitpoint_n.npy"), np.arange(n))


@pytest.mark.gpu
def test_b200_arm_dumps_the_state_its_last_step_left(gpu, tmp_path):
    """The dump equals the same rounds replayed here through the binding: counts and radii bit for bit, fp64 flux to the order of its sums."""
    P, W, S = 1 << 18, 1, 2
    d, D = _bench_with_dump(tmp_path, "--workload", "c2_bunny_chess", "--photons", str(P), "--warmup", str(W), "--steps", str(S), "--accum", "0",
                            "--cpu-photons", "0", "--e2e-rounds", "0")
    assert d["steps"] == S and d["config"]["hitpoints"] == len(D["hitpoint_r2"])
    with gpu.Context(0) as g:
        g.set_config(gpu.RenderConfig(width=1024, height=1024, hashsize=1000001), accum_mode=0)
        gpu.preset("c2_bunny_chess").build_into(g); g.commit()
        g.eye_pass(); g.build_grid()
        for k in range(W + S):
            g.photon_pass(k * P, P); g.round_update()
        hp = g.download_hitpoints(fields=("flux", "r2", "n"))
    assert np.array_equal(D["hitpoint_n"], hp["n"]) and hp["n"].sum() > 0
    assert np.array_equal(D["hitpoint_r2"], hp["r2"])
    assert np.allclose(D["hitpoint_flux"], hp["flux"], rtol=1e-9, atol=1e-9)


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode != 0           # no CPU fallback on the product path
    assert not r.stdout.strip()        # and no bench line
