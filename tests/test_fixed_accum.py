"""Fixed-point flux accumulators (accum_mode 2, include/cgrt.h): every accepted pair adds q = round-half-even(cf * 2^22) to int64 sums, so
flux, radii, counts and image are the same bits on every run, any launch split, any GPU count — and equal to the fixed-point oracle
(oracle_fixed/), which adds the same integers.

CPU: the oracle's fixed-point mode is independent of thread count and photon order, agrees with the fp64 oracle to the definition's
resolution, and ShardedRenderer over it with a gloo world of 2 equals world 1 bit for bit.
GPU: renders equal the oracle bit for bit (PPM and SPPM, c1-c4 and c3 at 1024^2; c1 without its Bezier vase, whose GPU solver matches the
reference statistically, not bit for bit — the vase scene is covered by the reproducibility tests); the crafted accept-boundary pairs of
tests/test_deposit_edges.py deposit exactly the oracle's q; renders are reproducible across repeats, call splits, call order, fenced
buffers and emulated ranks; out-of-range deposits and counts are refused; accum_mode outside {0, 1, 2} is refused.
Two GPUs: the library communicator, the peer exchange, torch host collectives and C++ render() equal one GPU bit for bit."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from tests.fixed_util import FixedOracleEngine, assert_same, observables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PPM, JITTER, CORNER = 0, 1, 2
ERR_INVALID, ERR_CAPACITY = -1, -4

# name -> (preset, max_tris, RenderConfig overrides)
CASES = {
    "c1": ("c1_spheres", None, dict(width=64, height=48)),
    "c1m": ("c1_mirror", None, dict(width=64, height=48)),
    "c1b": ("c1_spheres_bezier", None, dict(width=64, height=48)),
    "c2": ("c2_bunny_chess", None, dict(width=64, height=48)),
    "c3": ("c3_dragon_glass", 20000, dict(width=64, height=64)),
    "c4": ("c4_bump_dof", None, dict(width=64, height=36, use_dof=1, num_of_samples=4)),
}
ROUNDS, PHOTONS = 3, 30000


def case(name):
    from cgraytracing_b200 import RenderConfig, preset

    p, max_tris, kw = CASES[name]
    return preset(p, max_tris=max_tris), RenderConfig(update_mode=1, into_rule=1, **kw)


def threads():
    from oracle import binding as ob

    return min(16, ob.Oracle().max_threads())


def oracle_render(scene, cfg, sppm, rounds=ROUNDS, nph=PHOTONS, nthreads=1, reverse=False):
    from oracle_fixed.binding import FixedOracle

    o = FixedOracle(scene, cfg)
    if sppm:
        o.set_sppm(sppm)
    else:
        o.eye_pass(nthreads=threads())
    for r in range(rounds):
        if sppm:
            o.sppm_begin_round(r, threads())
        o.photon_pass(r * nph, nph, nthreads, reverse)
        o.round_update()
    out = observables(o, sppm, float(rounds * nph))
    assert o.error() == 0
    return out


def gpu_context(cg, scene, cfg, sppm, accum=2):
    g = cg.Context(0)
    g.set_config(cfg, accum_mode=accum)
    scene.build_into(g)
    g.commit()
    if sppm:
        g.set_sppm(sppm)
    return g


def gpu_render(cg, scene, cfg, sppm, rounds=ROUNDS, nph=PHOTONS, splits=1, reverse=False, accum=2):
    """The render on one GPU; each round's photons in `splits` calls, issued last range first when `reverse`."""
    with gpu_context(cg, scene, cfg, sppm, accum) as g:
        if not sppm:
            g.eye_pass()
            g.build_grid()
        for r in range(rounds):
            if sppm:
                g.sppm_begin_round(r)
            edges = np.linspace(0, nph, splits + 1).astype(np.int64)
            parts = [(r * nph + int(a), int(b - a)) for a, b in zip(edges, edges[1:])]
            for first, count in (parts[::-1] if reverse else parts):
                g.photon_pass(first, count)
            g.round_update()
        img, rgb8 = g.gather_image(float(rounds * nph), want_rgb8=True)
        out = observables(g, sppm, float(rounds * nph), rgb8)
        assert np.array_equal(out["img"], img)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_definition_is_float_product_and_half_even_rounding():
    """cf = ((float)f * (float)flux) * (float)(1/pi) in IEEE float; q = round-half-even(cf * 2^22) — against numpy's float32 arithmetic."""
    from oracle_fixed.binding import deposit_value

    rng = np.random.default_rng(5)
    f = np.concatenate([rng.uniform(0, 1, 20000), [0.0, 1.0, 0.15, 0.5, 1 / 3]])
    flux = np.concatenate([rng.uniform(0, 700 * 4 * np.pi, 20000), [1.0, 700 * 4 * 3.14159265358979, 2.5, 3.0, 7.0]])
    cf, q = deposit_value(f, flux)
    want = (f.astype(np.float32) * flux.astype(np.float32)) * np.float32(1.0 / 3.14159265358979)
    assert cf.dtype == np.float32 and np.array_equal(cf, want)
    x = cf.astype(np.float64) * 2.0 ** 22
    assert np.array_equal(q, np.rint(x).astype(np.int64))  # numpy's rint rounds half to even
    frac = x - np.floor(x)
    assert np.any(frac > 0.5) and np.any((frac > 0) & (frac < 0.5))  # both directions of the rounding occur
    big = cf >= 2.0
    assert np.all(q[big] == x[big])  # every value >= 2 is held exactly
    assert np.all(np.abs(q * 2.0 ** -22 - cf) <= 2.0 ** -23)


@pytest.mark.parametrize("sppm", [PPM, JITTER])
def test_oracle_is_independent_of_threads_and_photon_order(sppm):
    scene, cfg = case("c2")
    ref = oracle_render(scene, cfg, sppm, nthreads=1)
    assert ref["n"].sum() > 1000
    for nt, rev in ((4, False), (16, False), (1, True), (16, True)):
        assert_same(oracle_render(scene, cfg, sppm, nthreads=nt, reverse=rev), ref)


def test_oracle_agrees_with_fp64_within_resolution():
    """Same accepted counts as the fp64 U2 oracle; per hitpoint |sum cf - sum c| <= 6 * 2^-24 |sum c| + M 2^-23 (five float roundings
    of each positive term, then the fixed-point rounding of each)."""
    from oracle import binding as ob
    from oracle_fixed.binding import FixedOracle

    scene, cfg = case("c2")
    o64, ofx = ob.Oracle(scene, cfg), FixedOracle(scene, cfg)
    for o in (o64, ofx):
        o.eye_pass(nthreads=threads())
        o.photon_pass(0, 60000, threads())
    d64, m64 = o64.download_accum()
    dfx, mfx = ofx.download_accum()
    assert np.array_equal(mfx.astype(np.int64), m64.astype(np.int64)) and m64.sum() > 1000
    bound = 6 * 2.0 ** -24 * np.abs(d64) + mfx[:, None] * 2.0 ** -23
    assert np.all(np.abs(dfx - d64) <= bound)
    assert np.any(dfx != d64)
    for o in (o64, ofx):
        o.round_update()
    h64, hfx = o64.download_hitpoints(), ofx.download_hitpoints()
    assert np.array_equal(h64["n"], hfx["n"]) and np.array_equal(h64["r2"], hfx["r2"])


@pytest.mark.parametrize("name", ["c1b", "c1m", "c3", "c4"])
def test_oracle_photon_paths_are_the_oracles(name):
    """The fixed-point oracle traces photons with its own copy of the oracle's photon branch (only the deposit differs). Every path must
    stay the oracle's: the same segments, misses, diffuse hits, bucket probes, candidates, BVH work and accepted pairs per hitpoint, on
    scenes that reach every branch (Bezier, mirror, glass, displaced floor)."""
    from oracle import binding as ob
    from oracle_fixed.binding import FixedOracle

    scene, cfg = case(name)
    o64, ofx = ob.Oracle(scene, cfg), FixedOracle(scene, cfg)
    for o in (o64, ofx):
        o.eye_pass(nthreads=threads())
        o.photon_pass(0, 20000, threads())
    c64, cfx = o64.counters(), ofx.counters()
    assert c64 == cfx, {k: (c64[k], cfx[k]) for k in c64 if c64[k] != cfx[k]}
    assert c64["deposits"] > 0 and c64["photon_segments"] > c64["diffuse_hits"]
    assert np.array_equal(o64.download_accum()[1].astype(np.int64), ofx.download_accum()[1].astype(np.int64))


def _gloo_worker(rank, world, port, out, sppm):
    import torch.distributed as dist

    from cgraytracing_b200.distributed import ShardedRenderer

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        scene, cfg = case("c2")
        eng = FixedOracleEngine(scene, cfg, sppm)
        img = ShardedRenderer(eng, rank, world).render(cfg.height, ROUNDS, 5001)
        o = observables(eng.o, sppm, float(ROUNDS * 5001))
        assert np.array_equal(o["img"], img)
        np.savez(os.path.join(out, f"rank{rank}.npz"), **o)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("sppm", [PPM, JITTER, CORNER])
def test_sharded_oracle_two_ranks_equal_one_rank(tmp_path, sppm):
    import torch.multiprocessing as mp

    from cgraytracing_b200.distributed import ShardedRenderer

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path), sppm), nprocs=2, join=True)
    a, b = dict(np.load(tmp_path / "rank0.npz")), dict(np.load(tmp_path / "rank1.npz"))
    scene, cfg = case("c2")
    eng = FixedOracleEngine(scene, cfg, sppm)
    ShardedRenderer(eng).render(cfg.height, ROUNDS, 5001)
    one = observables(eng.o, sppm, float(ROUNDS * 5001))
    assert one["n"].sum() > 100
    assert_same(a, b)
    assert_same(a, one)


# ---------------------------------------------------------------------------------------------------------------------
# one GPU
# ---------------------------------------------------------------------------------------------------------------------
GPU_CASES = [("c1", PPM), ("c1m", PPM), ("c2", PPM), ("c3", PPM), ("c4", PPM), ("c2", JITTER), ("c2", CORNER), ("c4", JITTER), ("c4", CORNER)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,sppm", GPU_CASES)
def test_gpu_equals_oracle_bit_for_bit(gpu, name, sppm):
    scene, cfg = case(name)
    g = gpu_render(gpu, scene, cfg, sppm)
    o = oracle_render(scene, cfg, sppm, nthreads=threads())
    assert g["n"].sum() > 100
    assert_same(g, o, ("n", "r2", "flux", "img") + (() if sppm else ("pos", "key")))


@pytest.mark.gpu
def test_gpu_equals_oracle_c3_full_size(gpu):
    from cgraytracing_b200 import RenderConfig, preset

    scene, cfg = preset("c3_dragon_glass"), RenderConfig(width=1024, height=1024, update_mode=1, into_rule=1)
    g = gpu_render(gpu, scene, cfg, PPM, rounds=2, nph=400000)
    o = oracle_render(scene, cfg, PPM, rounds=2, nph=400000, nthreads=threads())
    assert g["n"].sum() > 10000
    assert_same(g, o, ("n", "r2", "flux", "img", "pos", "key"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ties", "rounding", "normals", "far", "faces", "dense"])
def test_gpu_crafted_pairs_deposit_the_oracle_q(gpu, name):
    """Pairs on the fp32 filters' accept boundary, thin-shell pairs of the fp64 test included: every accepted pair adds exactly q."""
    from oracle_fixed.binding import FixedOracle
    from tests import test_deposit_edges as de

    c = de.family(name)
    b = de.brute(c, de.HS)
    order = de.canonical(c, de.HS)
    o = FixedOracle(de.scene_for(c["scene"]), de.cfg_for(de.HS))
    o.import_hitpoints(c["hp"]["rec"][de.HS])
    de.oracle_trace(o, c)
    q = o.download_accum_i64()
    with de.gpu_context(gpu, c, de.HS, accum=2) as g:
        t = de.import_records(g, c["hp"]["rec"][de.HS])
        g.build_grid()
        de.gpu_trace(g, c)
        df, m = g.download_accum()
        del t
    assert np.array_equal(m.astype(np.int64), b["cnt"][order]) and np.array_equal(q[:, 3], b["cnt"][order])
    assert np.array_equal(df * 2.0 ** 22, q[:, :3].astype(np.float64)) and np.abs(q[:, :3]).max() < 2 ** 53
    region = de.float_decision(c, b)[1]
    if name != "dense":
        assert np.sum((region >= 2) & b["acc"]) > 0  # accepted pairs the fp32 filters leave to the fp64 test are among them


@pytest.mark.gpu
@pytest.mark.parametrize("name,sppm", [("c3", PPM), ("c3", JITTER), ("c1b", PPM)])
def test_gpu_render_is_reproducible(gpu, name, sppm):
    """The same render twice, each round's photons in 1 call, in 7 calls, and in 7 calls issued in reverse order: the same bits, 8-bit
    image included."""
    scene, cfg = case(name)
    ref = gpu_render(gpu, scene, cfg, sppm)
    assert_same(gpu_render(gpu, scene, cfg, sppm), ref)
    assert_same(gpu_render(gpu, scene, cfg, sppm, splits=7), ref)
    assert_same(gpu_render(gpu, scene, cfg, sppm, splits=7, reverse=True), ref)


@pytest.mark.gpu
def test_gpu_render_is_reproducible_with_fenced_buffers(gpu, tmp_path):
    """Under CGRT_GUARD=1 (every device buffer between fences, other addresses and sizes) the render is the same bits, no fence is hit."""
    scene, cfg = case("c3")
    ref = gpu_render(gpu, scene, cfg, PPM, splits=3)
    out = tmp_path / "guard.npz"
    env = dict(os.environ, CGRT_GUARD="1")
    subprocess.check_call([sys.executable, os.path.join(ROOT, "tests", "fixed_accum_worker.py"), "guard", str(out)], env=env, cwd=ROOT)
    got = dict(np.load(out))
    assert int(got.pop("damaged")) == 0
    assert_same(got, ref)


@pytest.mark.gpu
@pytest.mark.parametrize("sppm", [PPM, JITTER])
def test_gpu_two_contexts_as_ranks_equal_one_context(gpu, sppm):
    """Two contexts of one device play two ranks: row tiles (SPPM) or one eye pass each (PPM), disjoint photon ranges, the int64 sums added
    on the host. The result equals one context bit for bit."""
    import torch

    from cgraytracing_b200.distributed import HP_RECORD_DOUBLES, _DevArray, photon_shard, row_shard

    scene, cfg = case("c4")
    ranks = [gpu_context(gpu, scene, cfg, sppm) for _ in range(2)]
    try:
        if not sppm:
            for g in ranks:
                g.eye_pass()
                g.build_grid()
        for r in range(ROUNDS):
            if sppm:
                for k, g in enumerate(ranks):
                    g.sppm_eye_pass(r, *row_shard(cfg.height, k, 2))
                parts = []
                for g in ranks:
                    ptr, n = g.export_hitpoints_dev()
                    parts.append(torch.as_tensor(_DevArray(ptr, n * HP_RECORD_DOUBLES, "<f8"), device="cuda:0").view(n, HP_RECORD_DOUBLES))
                union = torch.cat(parts, 0)
                torch.cuda.synchronize()
                for g in ranks:
                    g.import_hitpoints_dev(union.data_ptr(), union.shape[0])
                    g.build_grid()
            for k, g in enumerate(ranks):
                g.photon_pass(*photon_shard(r, PHOTONS, k, 2))
            for g in ranks:
                g.synchronize()
            accs = []
            for g in ranks:
                ptr, n = g.accum_dev()
                accs.append(torch.as_tensor(_DevArray(ptr, n, "<i8"), device="cuda:0"))
            total = accs[0] + accs[1]
            for a in accs:
                a.copy_(total)
            torch.cuda.synchronize()
            for g in ranks:
                g.round_update()
        got = [observables(g, sppm, float(ROUNDS * PHOTONS)) for g in ranks]
    finally:
        for g in ranks:
            g.close()
    one = gpu_render(gpu, scene, cfg, sppm)
    assert_same(got[0], got[1])
    assert_same(got[0], one, ("n", "r2", "flux", "img"))


def hot_wall_scene():
    """walls_only with a back wall of colour 100: the deposit values of photons landing there exceed 2^16."""
    from cgraytracing_b200 import preset

    s = preset("walls_only")
    s.objects[3]["col"] = np.array([100.0, 100.0, 100.0])
    return s


def one_pixel_config():
    from cgraytracing_b200 import RenderConfig

    return RenderConfig(width=1, height=1, update_mode=1, into_rule=1)  # radius 200: the one hitpoint's sphere covers the room


CROWD = 48 << 20  # photons of one round: the single hitpoint accepts more than 2^24 of them


def refusal_run(cg, what, accum):
    """-> (status of the first synchronising call after round 1's update, the most photons one hitpoint accepted in the round as modes 0
    and 1 report them)."""
    from cgraytracing_b200 import RenderConfig

    if what == "value":
        scene, cfg, nph = hot_wall_scene(), RenderConfig(width=32, height=24, update_mode=1, into_rule=1), 200000
    else:
        scene, cfg, nph = case("c2")[0], one_pixel_config(), CROWD
    with gpu_context(cg, scene, cfg, PPM, accum) as g:
        g.eye_pass()
        g.build_grid()
        g.photon_pass(0, nph)
        mmax = float(g.download_accum()[1].max()) if accum != 2 else None
        g.round_update()
        rc = g.L.cgrt_synchronize(g.h)
        if rc == 0:
            img = g.gather_image(float(nph))
            assert np.all(np.isfinite(img))
            return rc, mmax
        msg = g.L.cgrt_last_error(g.h).decode()
        assert "fixed-point" in msg
        # the error stays raised: every later synchronising call reports it
        assert g.L.cgrt_synchronize(g.h) == rc
        with pytest.raises(cg.CgrtError):
            g.download_accum()
        return rc, None


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["value", "count"])
def test_gpu_out_of_range_is_refused(gpu, what):
    rc, _ = refusal_run(gpu, what, 2)
    assert rc == ERR_CAPACITY
    for accum in (0, 1):  # the other modes render the same scenes as before
        rc, mmax = refusal_run(gpu, what, accum)
        assert rc == 0
        if what == "count" and accum == 0:
            assert mmax > 2 ** 24  # the fixed-point refusal was for a real overflow of its count range


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [3, -1, 100])
def test_gpu_accum_mode_outside_range_is_invalid(gpu, mode):
    from cgraytracing_b200.binding import CgrtConfig

    import ctypes as C

    with gpu.Context(0) as g:
        k = CgrtConfig()
        g.L.cgrt_default_config(C.byref(k))
        k.accum_mode = mode
        assert g.L.cgrt_set_config(g.h, C.byref(k)) == ERR_INVALID
        assert "accum_mode" in g.L.cgrt_last_error(g.h).decode()
        k.accum_mode = 2
        assert g.L.cgrt_set_config(g.h, C.byref(k)) == 0
        assert g.L.cgrt_deposit_record_bytes(g.h) == 64


@pytest.mark.gpu
def test_gpu_version(gpu):
    assert gpu.load_library().cgrt_version() == 103


# ---------------------------------------------------------------------------------------------------------------------
# two GPUs
# ---------------------------------------------------------------------------------------------------------------------
def need_two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one box")


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["nccl", "peer", "torch"])
def test_two_gpus_equal_one_gpu(how):
    need_two_gpus()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port", "29541",
                        os.path.join(ROOT, "tests", "fixed_accum_worker.py"), "ranks", how], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert f"FIXED_RANKS_OK {how}" in r.stdout


@pytest.mark.gpu
def test_two_gpu_cpp_render_equals_one_gpu(tmp_path):
    """C++ render() with num_gpus = 2 (peer exchange and ncclAllReduce) prints and writes the one-GPU render's numbers and image bytes."""
    need_two_gpus()
    from cgraytracing_b200 import build

    build.build()
    host = os.path.join(ROOT, "cgraytracing_b200", "host")
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    subprocess.check_call(["make", "-C", host, "-s"], env=env)
    exe, assets = os.path.join(host, "example_main"), os.path.join(ROOT, "cgraytracing_b200", "assets")
    outs, imgs = [], []
    for tag, gpus, how in (("1", 1, "peer"), ("2p", 2, "peer"), ("2n", 2, "nccl")):
        p = tmp_path / f"o{tag}.ppm"
        o = subprocess.check_output([exe, "bunny", "160", "120", "60001", "3", str(p), assets, str(gpus), how, "off", "2"], text=True)
        outs.append(o.strip().splitlines()[-1])
        imgs.append(p.read_bytes())
    assert outs[0] == outs[1] == outs[2] and int(outs[0].split()[1]) > 0
    assert imgs[0] == imgs[1] == imgs[2]
