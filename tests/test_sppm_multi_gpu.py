"""Stochastic progressive photon mapping on several GPUs: every round's eye pass traced in row tiles, the records of the tiles all-gathered,
the same grid built from the union on every rank, disjoint photon ranges, one all-reduce of the round's accumulators before the per-pixel fold
(include/cgrt.h, cgrt_sppm_eye_pass).

CPU: cgraytracing_b200.distributed.ShardedRenderer in SPPM mode over the oracle's split round (sppm_eye_pass, record exchange, build_grid)
with gloo, world 2, against the oracle's one-call round (sppm_begin_round).
One GPU: the split round equals the one-call round; two contexts of one device emulate two ranks (tests/sppm_two_ranks.py) and equal one
context, also with fenced buffers; the refusals of the split round.
Two GPUs: torch.distributed worker (tests/sppm_worker.py) with the library's communicator and with host-driven collectives, and the C++
render() on two GPUs."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from oracle import binding as ob
from tests.util import OracleEngine

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
JITTER, CORNER = 1, 2


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the host logic of the sharded SPPM round over the reference, world 2 (gloo)
# ---------------------------------------------------------------------------------------------------------------------
VP = ("pos", "key", "hw", "r2")


class UnionEngine(OracleEngine):
    """OracleEngine that keeps every round's union of visible points."""

    def __init__(self, *args):
        super().__init__(*args)
        self.unions = []

    def build_grid(self):
        super().build_grid()
        self.unions.append(self.o.download_hitpoints(VP))


W, H, ROUNDS, PHOTONS = 64, 48, 3, 5001  # odd photon count: the remainder path


def _gloo_worker(rank, world, port, out, mode):
    import torch.distributed as dist

    from cgraytracing_b200 import RenderConfig, preset
    from cgraytracing_b200.distributed import ShardedRenderer

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = RenderConfig(width=W, height=H, update_mode=1, into_rule=1)
        eng = UnionEngine(preset("c2_bunny_chess"), cfg, mode)
        img = ShardedRenderer(eng, rank, world).render(H, ROUNDS, PHOTONS)
        px = eng.o.sppm_download_pixels()
        rounds = {f"{k}{r}": u[k] for r, u in enumerate(eng.unions) for k in u}
        np.savez(os.path.join(out, f"rank{rank}.npz"), img=img, n=px["n"], r2=px["r2"], tau=px["tau"], **rounds)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", [JITTER, CORNER], ids=["jitter", "corner"])
def test_two_ranks_equal_one_rank(tmp_path, mode):
    import torch.multiprocessing as mp

    from cgraytracing_b200 import RenderConfig, preset

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path), mode), nprocs=2, join=True)
    a, b = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    for k in a.files:  # the replicas stay bit-identical
        assert np.array_equal(a[k], b[k]), k
    # one rank: the reference's one-call round (eye pass and table together)
    cfg = RenderConfig(width=W, height=H, update_mode=1, into_rule=1)
    o = ob.Oracle(preset("c2_bunny_chess"), cfg)
    o.set_sppm(mode)
    for r in range(ROUNDS):
        o.sppm_begin_round(r)
        hp = o.download_hitpoints()
        assert len(hp["pos"]) > 0
        for k in VP:  # the union of the tiles is the round's visible-point set, in canonical order
            assert np.array_equal(a[f"{k}{r}"], hp[k]), (r, k)
        o.photon_pass(r * PHOTONS, PHOTONS)
        o.round_update()
    px = o.sppm_download_pixels()
    assert np.array_equal(a["n"], px["n"]) and a["n"].sum() > 1000  # integer counts, hence the radii: exact
    assert np.array_equal(a["r2"], px["r2"])
    # sums differ only by fp64 association (two partial sums added by the all-reduce)
    assert np.allclose(a["tau"], px["tau"], rtol=1e-12, atol=1e-14)
    assert np.allclose(a["img"], o.gather_image(float(ROUNDS * PHOTONS)), rtol=1e-12, atol=1e-14)


def test_pending_records_round_trip():
    """Export -> import of the pending visible points, then the table: the same round as the one-call sppm_begin_round."""
    from cgraytracing_b200 import RenderConfig, preset

    cfg = RenderConfig(width=40, height=30, update_mode=1, into_rule=1)
    s = preset("c2_bunny_chess")
    a, b = ob.Oracle(s, cfg), ob.Oracle(s, cfg)
    a.set_sppm(JITTER)
    b.set_sppm(JITTER)
    a.sppm_begin_round(5)
    lo, hi = 0, cfg.height
    b.sppm_eye_pass(5, 17, hi)  # the tiles in reverse order: the table's sort makes the order irrelevant
    rec = b.export_hitpoints()
    b.sppm_eye_pass(5, lo, 17)
    b.import_hitpoints(np.concatenate([rec, b.export_hitpoints()], 0))
    b.build_grid()
    ha, hb = a.download_hitpoints(), b.download_hitpoints()
    for k in VP:
        assert np.array_equal(ha[k], hb[k]), k
    assert len(ha["pos"]) >= cfg.width * cfg.height // 2


# ---------------------------------------------------------------------------------------------------------------------
# one GPU
# ---------------------------------------------------------------------------------------------------------------------
def _ctx(gpu, scene, cfg, mode, accum):
    from tests.sppm_two_ranks import sppm_context

    return sppm_context(gpu, scene, cfg, mode, accum)


def _flux_close(got, ref, n, accum):
    """fp64 sums in another order: 1e-9 relative. Float sums on both sides, each within the bound of tests/util.assert_flux_close of the
    exact sum: twice that bound apart at most."""
    got, ref = np.asarray(got).reshape(-1, 3), np.asarray(ref).reshape(-1, 3)
    if accum == 0:
        assert np.allclose(got, ref, rtol=1e-9, atol=1e-12)
    else:
        bound = 2 * (np.asarray(n, np.float64).reshape(-1)[:, None] + 8.0) * 2.0 ** -24 * np.abs(ref) + 1e-6
        err = np.abs(got - ref)
        assert np.all(err <= bound), float((err / bound).max())


def _pixels_close(got, ref, accum):
    _flux_close(got["tau"], ref["tau"], ref["n"], accum)


SPLIT = [("c2_bunny_chess", dict(width=96, height=72)), ("c4_bump_dof", dict(width=80, height=48, use_dof=1, num_of_samples=2))]


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("name,kw", SPLIT, ids=[p[0] for p in SPLIT])
def test_split_round_equals_one_call_round(gpu, name, kw, accum):
    """sppm_eye_pass(r, 0, H) + build_grid against sppm_begin_round(r), four rounds: every round's visible points and the final pixel n
    and R2 bit-equal. tau: the deposits are added by atomics, whose order is not repeatable from run to run (tests/test_sppm.py replays
    with the same bound), so it is compared to the accumulator type's precision."""
    R, N = 4, 20000
    s = gpu.preset(name)
    cfg = gpu.RenderConfig(**kw)
    with _ctx(gpu, s, cfg, JITTER, accum) as a, _ctx(gpu, s, cfg, JITTER, accum) as b:
        for r in range(R):
            a.sppm_begin_round(r)
            b.sppm_eye_pass(r, 0, cfg.height)
            b.build_grid()
            ha, hb = a.download_hitpoints(VP), b.download_hitpoints(VP)
            assert len(ha["pos"]) > 0
            for k in VP:
                assert np.array_equal(ha[k], hb[k]), (r, k)
            for g in (a, b):
                g.photon_pass(r * N, N)
                g.round_update()
        pa, pb = a.sppm_download_pixels(), b.sppm_download_pixels()
        assert np.array_equal(pa["n"], pb["n"]) and pa["n"].sum() > 0
        assert np.array_equal(pa["r2"], pb["r2"])
        _pixels_close(pb, pa, accum)


EMU = [("c1_spheres", None, dict(width=96, height=72)),
       ("c2_bunny_chess", None, dict(width=96, height=72)),
       ("c4_bump_dof", 20000, dict(width=80, height=48, use_dof=1, num_of_samples=2))]


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("mode", [JITTER, CORNER], ids=["jitter", "corner"])
@pytest.mark.parametrize("name,max_tris,kw", EMU, ids=[p[0] for p in EMU])
def test_two_contexts_equal_one_context(gpu, name, max_tris, kw, mode, accum):
    """Two contexts of one device as two ranks (tests/sppm_two_ranks.py) against one context over five rounds: every round's visible
    points bit-equal on both ranks, final pixel n and R2 bit-equal, tau and the image to the accumulator type's precision, and the two
    ranks' pixel statistics identical."""
    from tests.sppm_two_ranks import emulated_round

    R, N = 5, 20000
    s = gpu.preset(name, max_tris=max_tris)
    cfg = gpu.RenderConfig(**kw)
    with _ctx(gpu, s, cfg, mode, accum) as one, _ctx(gpu, s, cfg, mode, accum) as r0, _ctx(gpu, s, cfg, mode, accum) as r1:
        def check(ranks, r):
            ref = one.download_hitpoints(VP)
            assert len(ref["pos"]) > 0
            for g in ranks:
                got = g.download_hitpoints(VP)
                for k in VP:
                    assert np.array_equal(got[k], ref[k]), (r, k)

        for r in range(R):
            one.sppm_begin_round(r)
            emulated_round([r0, r1], r, N, cfg.height, on_grid=lambda ranks, r=r: check(ranks, r))
            one.photon_pass(r * N, N)
            one.round_update()
        p1, pa, pb = one.sppm_download_pixels(), r0.sppm_download_pixels(), r1.sppm_download_pixels()
        for k in ("n", "r2", "tau"):
            assert np.array_equal(pa[k], pb[k]), k
        assert np.array_equal(pa["n"], p1["n"]) and p1["n"].sum() > 0
        assert np.array_equal(pa["r2"], p1["r2"])
        _pixels_close(pa, p1, accum)
        ia, ib, i1 = r0.gather_image(float(R * N)), r1.gather_image(float(R * N)), one.gather_image(float(R * N))
        assert np.array_equal(ia, ib)
        _flux_close(ia, i1, p1["n"], accum)


@pytest.mark.gpu
def test_two_contexts_with_fenced_buffers():
    """The emulated two-rank rounds with CGRT_GUARD=1 (tests/sppm_two_ranks.py as a script): the per-round release and re-allocation of
    the tiles, the imported union, the grid and the accumulators write nothing outside their buffers."""
    env = dict(os.environ, CGRT_GUARD="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "sppm_two_ranks.py")], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "guard mode 1 damaged fence bytes 0" in r.stdout


@pytest.mark.gpu
def test_refusals_of_the_split_round(gpu):
    s = gpu.preset("walls_only")
    cfg = gpu.RenderConfig(width=32, height=24)
    with _ctx(gpu, s, cfg, JITTER, 0) as g:
        ptr, n = g.export_hitpoints_dev()
        with pytest.raises(gpu.CgrtError, match="SPPM"):
            g.import_hitpoints_dev(ptr, n)  # before any eye pass
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.allgather_hitpoints(1, 2)
        with pytest.raises(gpu.CgrtError, match="row range"):
            g.sppm_eye_pass(0, 10, 5)
        g.sppm_eye_pass(0, 0, 12)
        ptr, n = g.export_hitpoints_dev()
        assert n > 0
        import torch

        from tests.sppm_two_ranks import _dev

        rec = _dev(ptr, n * 12, "<f8").clone()
        torch.cuda.synchronize()
        g.import_hitpoints_dev(rec.data_ptr(), n)  # accepted between the eye pass and the grid
        g.build_grid()
        with pytest.raises(gpu.CgrtError, match="SPPM is on"):
            g.build_grid()  # twice in one round
        with pytest.raises(gpu.CgrtError, match="SPPM"):
            g.import_hitpoints_dev(rec.data_ptr(), n)
        with pytest.raises(gpu.CgrtError, match="multi-GPU SPPM"):
            g.allgather_hitpoints(1, 2)
        g.photon_pass(0, 1000)
        g.round_update()
        g.sppm_eye_pass(1, 5, 5)  # an empty tile: a rank without rows
        assert g.export_hitpoints_dev()[1] == 0
        g.build_grid()
        g.round_update()
    with gpu.Context(0) as g:
        g.set_config(cfg)
        s.build_into(g); g.commit()
        with pytest.raises(gpu.CgrtError, match="set_sppm"):
            g.sppm_eye_pass(0, 0, 24)  # SPPM is off


def _host_binary():
    from cgraytracing_b200 import build

    build.build()
    host = os.path.join(ROOT, "cgraytracing_b200", "host")
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    subprocess.check_call(["make", "-C", host, "-s"], env=env)
    return os.path.join(host, "example_main")


@pytest.mark.gpu
def test_cpp_render_refuses_sppm_with_peer_exchange(tmp_path):
    exe = _host_binary()
    r = subprocess.run([exe, "bunny", "32", "24", "1000", "1", str(tmp_path / "o.ppm"), os.path.join(ROOT, "cgraytracing_b200", "assets"), "2",
                        "peer", "jitter"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 1 and "peer exchange" in r.stderr, (r.returncode, r.stderr)


# ---------------------------------------------------------------------------------------------------------------------
# two GPUs
# ---------------------------------------------------------------------------------------------------------------------
def _need_two_gpus():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one box")


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("how", ["native", "host"])
def test_two_gpu_worker_equals_one_gpu(how, accum):
    _need_two_gpus()
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29537", os.path.join(ROOT, "tests", "sppm_worker.py"), str(accum), how],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert f"SPPM_OK {how} {accum}" in r.stdout


@pytest.mark.gpu
def test_cpp_render_on_two_gpus_equals_one(tmp_path):
    _need_two_gpus()
    exe = _host_binary()
    W, H = 96, 64
    out = {}
    for gpus in (1, 2):
        line = subprocess.check_output([exe, "bunny", str(W), str(H), "9000", "3", str(tmp_path / f"o{gpus}.ppm"),
                                        os.path.join(ROOT, "cgraytracing_b200", "assets"), str(gpus), "nccl", "jitter"], text=True, timeout=600).split()
        header = f"P6\n{W} {H}\n255\n".encode()
        ppm = (tmp_path / f"o{gpus}.ppm").read_bytes()
        assert ppm.startswith(header)
        out[gpus] = (int(line[0]), int(line[1]), np.frombuffer(ppm[len(header):], np.uint8).astype(int))
    assert out[1][0] == out[2][0] > 0 and out[1][1] == out[2][1] > 0  # visible points of the last round, deposits of all ranks
    assert np.abs(out[1][2] - out[2][2]).max() <= 1
