"""Stochastic progressive photon mapping (SPPM, include/cgrt.h cgrt_set_sppm): a new eye pass every round, statistics per pixel.

The CPU reference is the oracle's SPPM mode (oracle/oracle_capi.cpp, orc_set_sppm): the unchanged PPM oracle (oracle/ppm_oracle.hpp) driven
round by round with the SPPM camera, per-pixel statistics and fold.
CPU: corner mode on walls_only (one visible point per pixel) is the PPM oracle's estimator itself, bit for bit; the jittered camera stream
is deterministic per round, different between rounds and stays inside the pixel.
GPU: every round's visible points and the final pixel counts / radii equal the reference's bit for bit; corner mode equals the PPM path;
replay, steady device memory, fenced buffers, refusals, image statistics against PPM, and the C++ render()."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.util import assert_flux_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PASS_SPPM_EYE = 3
JITTER, CORNER = 1, 2


def pixel_index(hw, width):
    return hw[:, 0].astype(np.int64) * width + hw[:, 1]


def oracle_rounds(ob, scene, cfg, mode, rounds, nph, threads=1):
    """mode 0: the PPM oracle (one eye pass, per-hitpoint U2 updates); else the SPPM reference with that camera mode."""
    o = ob.Oracle(scene, cfg)
    if mode:
        o.set_sppm(mode)
    else:
        o.eye_pass(nthreads=threads)
    for r in range(rounds):
        if mode:
            o.sppm_begin_round(r, threads)
        o.photon_pass(r * nph, nph, threads)
        o.round_update()
    return o


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference against the PPM oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_corner_mode_on_walls_is_ppm_bit_for_bit(oracle_lib):
    from cgraytracing_b200 import RenderConfig, preset

    s = preset("walls_only")
    cfg = RenderConfig(width=64, height=48, update_mode=1, into_rule=1)
    R, N = 4, 12000
    ppm = oracle_rounds(oracle_lib, s, cfg, 0, R, N)
    spp = oracle_rounds(oracle_lib, s, cfg, CORNER, R, N)
    hp = ppm.download_hitpoints()
    px = spp.sppm_download_pixels()
    idx = pixel_index(hp["hw"], cfg.width)
    assert len(idx) == cfg.width * cfg.height and len(np.unique(idx)) == len(idx)  # exactly one visible point per pixel
    assert hp["n"].sum() > 0
    assert np.array_equal(px["n"].ravel()[idx], hp["n"])
    assert np.array_equal(px["r2"].ravel()[idx], hp["r2"])
    assert np.array_equal(px["tau"].reshape(-1, 3)[idx], hp["flux"])
    assert np.array_equal(spp.gather_image(float(R * N)), ppm.gather_image(float(R * N)))
    # and the last round's visible points are PPM's hitpoints at the radius the round used
    last = spp.download_hitpoints()
    assert np.array_equal(last["pos"], hp["pos"]) and np.array_equal(last["key"], hp["key"]) and np.array_equal(last["hw"], hp["hw"])


def test_jitter_stream_is_per_round_and_inside_the_pixel(oracle_lib):
    from cgraytracing_b200 import RenderConfig, preset

    ob = oracle_lib
    s = preset("walls_only")
    cfg = RenderConfig(width=40, height=30, update_mode=1, into_rule=1)
    o = ob.Oracle(s, cfg)
    o.set_sppm(JITTER)
    o.sppm_begin_round(7)
    a = o.download_hitpoints()
    o.sppm_begin_round(7)
    b = o.download_hitpoints()
    o.sppm_begin_round(8)
    c = o.download_hitpoints()
    for k in ("pos", "key", "hw", "r2"):
        assert np.array_equal(a[k], b[k]), k  # the same round traced twice: identical visible points
    ia, ic = pixel_index(a["hw"], cfg.width), pixel_index(c["hw"], cfg.width)
    pa = np.zeros((cfg.width * cfg.height, 3)); pa[ia] = a["pos"]
    pc = np.zeros((cfg.width * cfg.height, 3)); pc[ic] = c["pos"]
    assert (np.abs(pa - pc).max(axis=1) > 0).mean() > 0.99  # another round: another point in (nearly) every pixel
    # the jitter of round r, pixel (h, w) is the first two draws of Philox (seed, PASS_SPPM_EYE, path, r): recompute it and check that the
    # visible point lies on that camera ray, and that the jitter is inside [0,1)^2
    seed = cfg.seed
    rng = np.random.default_rng(0)
    cam = np.array(cfg.camorg)
    for p in rng.choice(len(ia), 50, replace=False):
        h, w = a["hw"][p]
        path = int(h) * cfg.width + int(w)
        words = ob.philox([path & 0xFFFFFFFF, path >> 32, 7, 0], [seed & 0xFFFFFFFF, ((seed >> 32) + PASS_SPPM_EYE) & 0xFFFFFFFF])
        ux, uy = (words[:2] >> 1).astype(np.float64) * (1.0 / 2147483648.0)
        assert 0.0 <= ux < 1.0 and 0.0 <= uy < 1.0
        x = (2.0 * ((w + ux) / cfg.width) - 1) * 10.0
        y = (2.0 * ((h + uy) / cfg.height) - 1) * 10.0 * cfg.height / cfg.width
        d = np.array([x, y, 0.0]) - cam
        d /= np.linalg.norm(d)
        v = a["pos"][p] - cam
        assert np.linalg.norm(np.cross(v / np.linalg.norm(v), d)) < 1e-9  # the point is on the ray through (w + ux, h + uy)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def gpu_sppm(gpu, scene, cfg, mode, accum=0):
    g = gpu.Context(0)
    g.set_config(cfg, accum_mode=accum)
    scene.build_into(g)
    g.commit()
    g.set_sppm(mode)
    return g


PARITY = [("c1_spheres", None, dict(width=96, height=72)),
          ("c2_bunny_chess", None, dict(width=96, height=72)),
          ("c4_bump_dof", 20000, dict(width=80, height=48, use_dof=1, num_of_samples=2))]


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("mode", [JITTER, CORNER])
@pytest.mark.parametrize("name,max_tris,kw", PARITY, ids=[p[0] for p in PARITY])
def test_rounds_match_oracle(gpu, oracle_lib, name, max_tris, kw, mode, accum):
    """Five rounds against the oracle's SPPM mode: each round's visible points (pos, key, r2, pixel) bit-equal, and the round's accepted
    photons per visible point equal; final pixel n and R2 bit-equal; tau and the image within the accumulator type's bounds
    (tests/util.assert_flux_close)."""
    R, N = 5, 20000
    s = gpu.preset(name, max_tris=max_tris)
    cfg = gpu.RenderConfig(update_mode=1, into_rule=1, **kw)
    o = oracle_lib.Oracle(s, cfg)
    o.set_sppm(mode)
    th = max(1, len(os.sched_getaffinity(0)))
    with gpu_sppm(gpu, s, cfg, mode, accum) as g:
        for r in range(R):
            g.sppm_begin_round(r)
            o.sppm_begin_round(r, th)
            a, b = g.download_hitpoints(), o.download_hitpoints()
            assert len(a["pos"]) == len(b["pos"]) > 0, r
            for k in ("pos", "key", "r2", "hw"):
                assert np.array_equal(a[k], b[k]), (r, k)
            g.photon_pass(r * N, N)
            o.photon_pass(r * N, N, th)
            _, gm = g.download_accum()
            assert np.array_equal(gm.astype(np.int64), o.download_accum()[1].astype(np.int64)), r
            g.round_update()
            o.round_update()
        pg, po = g.sppm_download_pixels(), o.sppm_download_pixels()
        assert po["n"].sum() > 0
        assert np.array_equal(pg["n"], po["n"])
        assert np.array_equal(pg["r2"], po["r2"])
        n = po["n"].reshape(-1)
        assert_flux_close(pg["tau"].reshape(-1, 3), po["tau"].reshape(-1, 3), n, accum)
        img, oimg = g.gather_image(float(R * N)), o.gather_image(float(R * N))
        assert_flux_close(img.reshape(-1, 3), oimg.reshape(-1, 3), n, accum)


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
def test_corner_mode_equals_ppm_path(gpu, accum):
    """walls_only has one visible point per pixel: corner-mode SPPM is the PPM path itself — n and r2 bit for bit, the image to the
    rounding of the accumulators' addition order."""
    R, N = 4, 40000
    s = gpu.preset("walls_only")
    cfg = gpu.RenderConfig(width=128, height=96)
    with gpu.Context(0) as p, gpu_sppm(gpu, s, cfg, CORNER, accum) as g:
        p.set_config(cfg, accum_mode=accum)
        s.build_into(p); p.commit()
        p.eye_pass(); p.build_grid()
        for r in range(R):
            p.photon_pass(r * N, N); p.round_update()
            g.sppm_begin_round(r); g.photon_pass(r * N, N); g.round_update()
        hp = p.download_hitpoints()
        px = g.sppm_download_pixels()
        idx = pixel_index(hp["hw"], cfg.width)
        assert len(np.unique(idx)) == len(idx) == cfg.width * cfg.height and hp["n"].sum() > 0
        assert np.array_equal(px["n"].ravel()[idx], hp["n"])
        assert np.array_equal(px["r2"].ravel()[idx], hp["r2"])
        a, b = g.gather_image(float(R * N)), p.gather_image(float(R * N))
        if accum == 0:
            assert np.allclose(a, b, rtol=1e-9, atol=1e-12)
        else:  # float sums in another order on each side: the bound of assert_flux_close, twice
            n = px["n"].reshape(-1)[:, None].astype(np.float64)
            assert np.all(np.abs(a - b).reshape(-1, 3) <= 2 * (n + 8.0) * 2.0 ** -24 * np.abs(b).reshape(-1, 3) + 1e-9)


@pytest.mark.gpu
def test_replay_gives_the_same_pixels(gpu):
    """A new context replaying rounds 0..K reaches the same pixel state (fp64 accumulators: n, R2 bit-equal, tau to atomic order)."""
    K, N = 4, 30000
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=96, height=72)
    out = []
    for _ in range(2):
        with gpu_sppm(gpu, s, cfg, JITTER) as g:
            for r in range(K + 1):
                g.sppm_begin_round(r); g.photon_pass(r * N, N); g.round_update()
            out.append(g.sppm_download_pixels())
    assert np.array_equal(out[0]["n"], out[1]["n"]) and out[0]["n"].sum() > 0
    assert np.array_equal(out[0]["r2"], out[1]["r2"])
    assert np.allclose(out[0]["tau"], out[1]["tau"], rtol=1e-9, atol=1e-12)


@pytest.mark.gpu
def test_device_memory_reaches_a_steady_state(gpu):
    """Free device memory after round 3 equals free memory after round 30 within 64 MiB (a pool chunk): every round releases the
    last round's visible points and grid and asks for the same buffer sizes again."""
    import torch

    N = 30000
    s = gpu.preset("c3_dragon_glass", max_tris=20000)
    cfg = gpu.RenderConfig(width=160, height=120)
    free = {}
    with gpu_sppm(gpu, s, cfg, JITTER, accum=1) as g:
        for r in range(31):
            g.sppm_begin_round(r); g.photon_pass(r * N, N); g.round_update()
            if r in (3, 30):
                g.synchronize()
                free[r] = torch.cuda.mem_get_info(0)[0]
    assert abs(free[3] - free[30]) <= 64 << 20, (free[3] - free[30]) / 2**20


@pytest.mark.gpu
def test_no_out_of_bounds_writes_with_fenced_buffers():
    """SPPM rounds over every scene family, both camera modes and both accumulator types with CGRT_GUARD=1 (tools/sppm_guard_probe.py)."""
    env = dict(os.environ, CGRT_GUARD="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sppm_guard_probe.py")], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "guard mode 1 damaged fence bytes 0" in r.stdout


@pytest.mark.gpu
def test_refusals(gpu):
    s = gpu.preset("walls_only")
    cfg = gpu.RenderConfig(width=32, height=24)
    with gpu.Context(0) as g:
        g.set_config(cfg)
        s.build_into(g)
        with pytest.raises(gpu.CgrtError, match="commit"):
            g.set_sppm(JITTER)
        g.commit()
        with pytest.raises(gpu.CgrtError, match="set_sppm"):
            g.sppm_begin_round(0)  # SPPM is off
        with pytest.raises(gpu.CgrtError, match="mode"):
            g.set_sppm(3)
        g.eye_pass()
        with pytest.raises(gpu.CgrtError, match="before any eye pass"):
            g.set_sppm(JITTER)
    with gpu.Context(0) as g:
        g.set_config(gpu.RenderConfig(width=32, height=24, update_mode=0))
        s.build_into(g); g.commit()
        with pytest.raises(gpu.CgrtError, match="per-round update"):
            g.set_sppm(JITTER)
    with gpu.Context(0) as g:
        g.set_config(cfg)
        s.build_into(g); g.commit()
        g.eye_pass(); g.build_grid()
        with pytest.raises(gpu.CgrtError, match="before any eye pass"):
            g.set_sppm(CORNER)
    with gpu_sppm(gpu, s, cfg, JITTER) as g:
        with pytest.raises(gpu.CgrtError, match="SPPM is on"):
            g.eye_pass()
        with pytest.raises(gpu.CgrtError, match="SPPM is on"):
            g.build_grid()
        with pytest.raises(gpu.CgrtError, match="SPPM"):
            g.set_config(cfg)
        g.sppm_begin_round(0)
        ptr, n = g.export_hitpoints_dev()
        with pytest.raises(gpu.CgrtError, match="SPPM"):
            g.import_hitpoints_dev(ptr, n)
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.set_comm(1, 2)  # checked before the communicator is ever used
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.allgather_hitpoints(1, 2)
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.peer_attach(0, 1, [bytes(128)])
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.peer_export()
        o = np.array([[0.0, 0.0, -10.0]]); d = np.array([[0.0, 0.0, 1.0]]); w = np.ones((1, 3))
        with pytest.raises(gpu.CgrtError, match="SPPM is on"):
            g.trace(o, d, w, True, x=[0], y=[0])
        g.trace(o, d, w * 100.0, False, first_index=1 << 40)  # photons are still welcome
        g.photon_pass(0, 1000); g.round_update()
        assert g.sppm_download_pixels()["n"].sum() > 0


# ---------------------------------------------------------------------------------------------------------------------
# image statistics
# ---------------------------------------------------------------------------------------------------------------------
def render(gpu, name, kw, mode, rounds, nph, max_tris=None):
    """mode 0: PPM (one eye pass); else SPPM. -> linear image after `rounds` rounds of `nph` photons (float accumulators)."""
    s = gpu.preset(name, max_tris=max_tris)
    cfg = gpu.RenderConfig(**kw)
    with gpu.Context(0) as g:
        g.set_config(cfg, accum_mode=1)
        s.build_into(g); g.commit()
        if mode:
            g.set_sppm(mode)
        else:
            g.eye_pass(); g.build_grid()
        for r in range(rounds):
            if mode:
                g.sppm_begin_round(r)
            g.photon_pass(r * nph, nph); g.round_update()
        return g.gather_image(float(rounds * nph))


def box8(img):
    h, w = img.shape[0] // 8 * 8, img.shape[1] // 8 * 8
    return img[:h, :w].reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3))


def sppm_vs_ppm_stats(gpu, name):
    """-> (max relative difference of the per-channel means, 8x8-box RMSE relative to the mean) of SPPM (jitter) against PPM at equal
    photon budget."""
    kw = dict(width=256, height=256)
    a = render(gpu, name, kw, JITTER, 16, 1 << 20)
    b = render(gpu, name, kw, 0, 16, 1 << 20)
    ma, mb = a.mean(axis=(0, 1)), b.mean(axis=(0, 1))
    dmean = float(np.max(np.abs(ma - mb) / mb))
    rmse = float(np.sqrt(np.mean((box8(a) - box8(b)) ** 2)) / b.mean())
    return dmean, rmse


def dof_errors(gpu):
    """-> (RMSE of SPPM, RMSE of PPM with one sample) against a long SPPM render of the DOF scene, relative to its mean."""
    kw = dict(width=160, height=96, use_dof=1, num_of_samples=1)
    ref = render(gpu, "c4_bump_dof", kw, JITTER, 256, 1 << 20)
    a = render(gpu, "c4_bump_dof", kw, JITTER, 16, 1 << 20)
    b = render(gpu, "c4_bump_dof", kw, 0, 16, 1 << 20)
    e = lambda x: float(np.sqrt(np.mean((x - ref) ** 2)) / ref.mean())
    return e(a), e(b)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c3_dragon_glass", "c1_spheres"])
def test_sppm_and_ppm_images_agree(gpu, name):
    """16 rounds x 1 Mi photons at 256x256, float accumulators. SPPM converges to the pixel-area average and PPM to the pixel-corner value,
    so they agree in the per-channel means and at a coarse scale; at this budget the 8x8-box RMSE is mostly the photon noise of the two
    renders. Measured on one B200 (NVIDIA B200, 1000 W power limit): c3 means within 0.46 %, 8x8-box RMSE 22.5 % of the mean; c1 0.47 %
    and 21.8 %. Bounds: means 2.5x, RMSE 1.5x the measured values (the inputs are seeded: only the order of the float additions moves)."""
    dmean, rmse = sppm_vs_ppm_stats(gpu, name)
    lim = {"c3_dragon_glass": (0.0115, 0.34), "c1_spheres": (0.0115, 0.33)}[name]
    assert dmean < lim[0] and rmse < lim[1], (dmean, rmse)


@pytest.mark.gpu
def test_sppm_dof_converges_where_ppm_cannot(gpu):
    """Depth of field at 160x96: PPM with one sample keeps the lens sample of its single eye pass, SPPM draws a new one every round.
    At the same budget (16 rounds x 1 Mi photons) SPPM is closer to a long SPPM render (256 rounds). Measured on one B200 (1000 W power
    limit): RMSE 0.060 (SPPM) against 0.182 (PPM) of the long render's mean, a ratio of 0.33. Bound: SPPM below 0.5x PPM's error."""
    e_sppm, e_ppm = dof_errors(gpu)
    assert e_sppm < 0.5 * e_ppm, (e_sppm, e_ppm)


# ---------------------------------------------------------------------------------------------------------------------
# C++ host API
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode,mode_id", [("jitter", JITTER), ("corner", CORNER)])
def test_cpp_render_equals_python_binding(gpu, tmp_path, mode, mode_id):
    """render() with RenderOptions::sppm (example_main's trailing mode argument) == the same rounds through the Python binding."""
    from cgraytracing_b200 import build

    build.build()
    host = os.path.join(ROOT, "cgraytracing_b200", "host")
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    subprocess.check_call(["make", "-C", host, "-s"], env=env)
    W, H, NPH, ROUNDS = 96, 64, 9000, 3
    out = subprocess.check_output([os.path.join(host, "example_main"), "bunny", str(W), str(H), str(NPH), str(ROUNDS), str(tmp_path / "o.ppm"),
                                   os.path.join(ROOT, "cgraytracing_b200", "assets"), "1", "nccl", mode], text=True).split()
    with gpu_sppm(gpu, gpu.preset("c2_bunny_chess"), gpu.RenderConfig(width=W, height=H), mode_id) as g:
        done = 0
        for r in range(ROUNDS):
            n = NPH // ROUNDS + (1 if r < NPH % ROUNDS else 0)
            g.sppm_begin_round(r); g.photon_pass(done, n); g.round_update()
            done += n
        img, rgb8 = g.gather_image(float(NPH), want_rgb8=True)
        k = g.counters()
    assert int(out[0]) == k["hitpoints"] > 0 and int(out[1]) == k["deposits"] > 0
    ppm = (tmp_path / "o.ppm").read_bytes()
    header = f"P6\n{W} {H}\n255\n".encode()
    assert ppm.startswith(header)
    got8 = np.frombuffer(ppm[len(header):], np.uint8).reshape(H, W, 3)
    assert np.abs(got8.astype(int) - rgb8.astype(int)).max() <= 1
