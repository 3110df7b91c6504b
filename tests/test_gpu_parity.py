"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same seeded inputs.
Bars (BASELINE.md section 5): cell keys / sorted order bit-exact; t and normals <= 1e-5 relative (we assert bit-exact,
the stronger statement, where the arithmetic is the same); accepted-photon counts equal; flux within 1e-9 (fp64 atomic order)."""
import numpy as np
import pytest

from tests.util import camera_rays, random_rays, rel_err

pytestmark = pytest.mark.gpu

T_TOL = 1e-5  # relative, north_star


def make(gpu, ob, name, cfg_kw=None, max_tris=None):
    cfg = gpu.RenderConfig(**(cfg_kw or {}))
    s = gpu.preset(name, max_tris=max_tris)
    return s, cfg, gpu.Context(0, s, cfg), ob.Oracle(s, cfg)


def test_hash_keys_bit_exact(gpu, oracle_lib):
    ob = oracle_lib
    rng = np.random.default_rng(3)
    pos = rng.uniform(-40, 60, (200000, 3))
    pos[:1000] = np.round(pos[:1000] * 4) / 4  # cell-boundary-ish values
    with gpu.Context(0) as g:
        for h in (512, 768, 1024, 1080, 4096):
            k, ixyz = g.hash_keys(pos, 1000001, 200.0 / h)
            ok, oixyz = ob.hash_keys(pos, 1000001, 200.0 / h)
            assert np.array_equal(ixyz, oixyz)
            assert np.array_equal(k, ok)
        k, _ = g.hash_keys(pos, 16777259, 200.0 / 4096)
        ok, _ = ob.hash_keys(pos, 16777259, 200.0 / 4096)
        assert np.array_equal(k, ok)


def test_radix_sort_stable(gpu):
    rng = np.random.default_rng(4)
    with gpu.Context(0) as g:
        for n, bits in ((1, 8), (255, 16), (4096, 24), (100003, 40), (1 << 20, 52)):
            keys = rng.integers(0, 1 << bits, n, dtype=np.uint64)
            keys[: n // 3] = keys[0]  # many duplicates: stability matters
            out, perm = g.radix_sort(keys, bits)
            ref = np.argsort(keys, kind="stable")
            assert np.array_equal(perm, ref.astype(np.uint32))
            assert np.array_equal(out, keys[ref])


def test_philox_sampling_matches_oracle(gpu, oracle_lib):
    ob = oracle_lib
    with gpu.Context(0) as g:
        for path in (0, 1, 12345678901, 2**40 + 17):
            for what, aux in ((0, (0, 0, 0)), (1, (0.3, -0.8, 0.52)), (2, (1.5, 0, 0)), (3, (0, 0, 0))):
                a = g.sample(20261018, 1, path, 3, what, aux)
                b = ob.sample(20261018, 1, path, 3, what, aux)
                assert np.array_equal(a, b), (path, what)


@pytest.mark.parametrize("name,max_tris", [("c1_spheres", None), ("c2_bunny_chess", None), ("c3_dragon_glass", 20000), ("c4_bump_dof", None),
                                           ("default_bump", 20000)])
def test_intersect_batch_matches_oracle(gpu, oracle_lib, name, max_tris):
    s, cfg, g, o = make(gpu, oracle_lib, name, dict(into_rule=1), max_tris)
    with g:
        for org, dr in (random_rays(40000, 5), camera_rays(1024, 768, 7)):
            a = g.intersect_batch(org, dr)
            b = o.intersect_batch(org, dr)
            assert np.array_equal(a["obj"], b["obj"])
            hit = b["obj"] >= 0
            assert hit.mean() > 0.9
            # north-star bar
            assert rel_err(a["t"][hit], b["t"][hit]).max() <= T_TOL
            assert np.abs(a["nrm"][hit] - b["nrm"][hit]).max() <= T_TOL
            # what we actually achieve: the same fp64 arithmetic -> identical bits (ties between coplanar triangles aside)
            same_prim = a["prim"] == b["prim"]
            assert same_prim.mean() > 0.999
            assert np.array_equal(a["t"][same_prim], b["t"][same_prim])
            assert np.array_equal(a["nrm"][same_prim], b["nrm"][same_prim])
            assert np.array_equal(a["into"][same_prim], b["into"][same_prim])


def test_bvh_equals_brute_force(gpu, oracle_lib):
    """Property: LBVH closest hit == brute force over all triangles (SURVEY section 4, item 3)."""
    s, cfg, g, o = make(gpu, oracle_lib, "c3_dragon_glass", dict(into_rule=1), 30000)
    mesh_id = len(s.objects) - 1
    with g:
        org, dr = random_rays(3000, 9)
        a = g.intersect_batch(org, dr)
        hit, ln, tri = o.mesh_brute(mesh_id, org, dr)
        on_mesh = a["obj"] == mesh_id
        # every GPU mesh hit is the brute-force closest triangle
        assert np.array_equal(a["t"][on_mesh], ln[on_mesh])
        # and where brute force hits the mesh closer than anything else the GPU reports the mesh
        walls = o.intersect_batch(org, dr)
        assert np.array_equal(on_mesh, walls["obj"] == mesh_id)


def test_bump_heightfield_triangles_bit_exact(gpu, oracle_lib):
    s, cfg, g, o = make(gpu, oracle_lib, "c4_bump_dof")
    with g:
        t = g.object_triangles(0)
        assert len(t) == 146744
        assert np.array_equal(t, o.bump_triangles(0))


def test_surface_color_matches_oracle(gpu, oracle_lib):
    s, cfg, g, o = make(gpu, oracle_lib, "c2_bunny_chess")
    rng = np.random.default_rng(6)
    pos = np.stack([rng.uniform(-25, 25, 50000), np.full(50000, -20.0), rng.uniform(-5, 45, 50000)], -1)
    with g:
        assert np.array_equal(g.surface_color(0, pos), o.surface_color(0, pos))
        assert np.array_equal(g.surface_color(1, pos), o.surface_color(1, pos))


@pytest.mark.parametrize("name,max_tris,W,H", [("c1_spheres", None, 256, 192), ("c2_bunny_chess", None, 256, 256), ("c3_dragon_glass", 30000, 192, 192),
                                               ("default_bump", 20000, 128, 96)])
def test_eye_pass_hitpoints_bit_exact(gpu, oracle_lib, name, max_tris, W, H):
    """Hitpoints, their cell keys and their sorted (canonical) order equal the oracle's bit for bit."""
    s, cfg, g, o = make(gpu, oracle_lib, name, dict(width=W, height=H, into_rule=1, update_mode=1), max_tris)
    with g:
        g.eye_pass()
        g.build_grid()
        a = g.download_hitpoints()
        o.eye_pass()
        b = o.download_hitpoints()
        assert len(a["pos"]) == len(b["pos"]) > 0
        assert np.array_equal(a["key"], b["key"])
        assert np.array_equal(a["hw"], b["hw"])
        for k in ("pos", "normal", "f", "r2"):
            assert np.array_equal(a[k], b[k]), k
        # creation sequence (path*16+dfs code) orders exactly like the oracle's insertion counter inside every bucket
        assert np.array_equal(a["seq"], (b["path"] * 16 + b["code"]).astype(np.uint32))
        cs = g.download_grid()
        assert cs[0] == 0 and cs[-1] == len(a["key"])
        counts = np.bincount(b["key"], minlength=cfg.hashsize)
        assert np.array_equal(np.diff(cs.astype(np.int64)), counts)
        assert g.counters()["eye_segments"] == o.counters()["eye_segments"]


@pytest.mark.parametrize("cull", [1, 0])
@pytest.mark.parametrize("name,max_tris", [("c1_spheres", None), ("c2_bunny_chess", None), ("c3_dragon_glass", 30000), ("default_bump", 20000)])
def test_photon_rounds_match_oracle(gpu, oracle_lib, name, max_tris, cull):
    """Two U2 rounds with the same Philox streams: integer counts equal, flux equal to fp64-atomic-order rounding, image equal.
    cull = 0 also makes the GPU scan exactly the candidates the reference scans (counters.candidates equal); with the reach-map
    culling on (default) the unreachable hits are skipped: fewer candidates, identical deposits."""
    W, H, NPH = 160, 120, 30000
    s, cfg, g, o = make(gpu, oracle_lib, name, dict(width=W, height=H, into_rule=1, update_mode=1), max_tris)
    with g:
        g.set_culling(bool(cull))
        g.eye_pass(); g.build_grid()
        o.eye_pass()
        for rnd in range(2):
            g.photon_pass(rnd * NPH, NPH)
            o.photon_pass(rnd * NPH, NPH)
            df, m = g.download_accum()
            odf, om = o.download_accum()
            assert np.array_equal(m.astype(np.int64), om.astype(np.int64))
            assert np.allclose(df, odf, rtol=1e-9, atol=1e-12)
            g.round_update(); o.round_update()
        a = g.download_hitpoints(); b = o.download_hitpoints()
        assert np.array_equal(a["n"], b["n"])
        assert np.array_equal(a["r2"], b["r2"])
        assert np.allclose(a["flux"], b["flux"], rtol=1e-9, atol=1e-12)
        img = g.gather_image(2.0 * NPH)
        assert np.allclose(img, o.gather_image(2.0 * NPH), rtol=1e-9, atol=1e-12)
        gc, oc = g.counters(), o.counters()
        for k in ("photon_segments", "diffuse_hits", "deposits"):
            assert gc[k] == oc[k], k
        assert gc["candidates"] == oc["candidates"] if not cull else 0 < gc["candidates"] <= oc["candidates"]


def test_photon_shards_are_invariant(gpu, oracle_lib):
    """Photons [0,N) in one call == two disjoint sub-ranges (what two GPUs would trace) summed: same counts, same flux."""
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=128, height=96)
    N = 20000
    with gpu.Context(0, s, cfg) as g1, gpu.Context(0, s, cfg) as g2:
        for g in (g1, g2):
            g.eye_pass(); g.build_grid()
        g1.photon_pass(0, N)
        g2.photon_pass(N // 2, N - N // 2)
        g2.photon_pass(0, N // 2)
        d1, m1 = g1.download_accum(); d2, m2 = g2.download_accum()
        assert np.array_equal(m1, m2)
        assert np.allclose(d1, d2, rtol=1e-9, atol=1e-12)


def test_f32_accumulators_close_to_f64(gpu):
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=128, height=96)
    with gpu.Context(0) as g64, gpu.Context(0) as g32:
        for g, mode in ((g64, 0), (g32, 1)):
            g.set_config(cfg, accum_mode=mode)
            s.build_into(g); g.commit()
            g.eye_pass(); g.build_grid(); g.photon_pass(0, 30000)
        d64, m64 = g64.download_accum(); d32, m32 = g32.download_accum()
        assert np.array_equal(m64, m32)
        assert np.allclose(d32, d64, rtol=1e-4, atol=1e-3)


def test_tile_sharded_eye_pass_equals_unsharded(gpu):
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=128, height=96)
    with gpu.Context(0, s, cfg) as g1, gpu.Context(0, s, cfg) as g2:
        g1.eye_pass(); g1.build_grid()
        g2.eye_pass(48, 96); g2.eye_pass(0, 48); g2.build_grid()
        a, b = g1.download_hitpoints(), g2.download_hitpoints()
        for k in a:
            assert np.array_equal(a[k], b[k]), k


def test_empty_and_error_paths(gpu):
    with gpu.Context(0) as g:
        g.set_config(gpu.RenderConfig(width=16, height=16))
        with pytest.raises(gpu.CgrtError):
            g.eye_pass()  # scene not committed
        g.commit()  # an empty scene is legal: every ray misses
        g.eye_pass(); g.build_grid()
        assert g.num_hitpoints() == 0
        g.photon_pass(0, 100)
        g.round_update()
        assert np.all(g.gather_image(100.0) == 0)
        with pytest.raises(gpu.CgrtError):
            g.commit()


# ---------------------------------------------------------------------------------------------------------------------
# against the committed outputs of the unmodified reference (tests/golden/ref_golden.npz, made by tests/golden/make_golden.py)
# ---------------------------------------------------------------------------------------------------------------------
import os  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.npz")


def test_hash_keys_vs_reference_golden(gpu):
    G = np.load(GOLDEN)
    with gpu.Context(0) as g:
        for h in (512, 768, 1024, 1080, 4096):
            k, ixyz = g.hash_keys(G["hash__pos"], 1000001, 200.0 / h)
            assert np.array_equal(k, G[f"hash_{h}__key"]) and np.array_equal(ixyz, G[f"hash_{h}__ixyz"])


@pytest.mark.parametrize("name", ["c1_spheres", "c2_bunny_chess", "c3_dragon_glass", "default_bump", "c4_bump_dof"])
def test_closest_hit_vs_reference_golden(gpu, name):
    """t, face-forwarded normal, object id of the reference's own closest-hit loop (main.cpp:50-76) on dumped ray batches.
    The raw mesh normal / `into` flag follow the GPU's winding rule, compared separately (SURVEY Q8)."""
    G = np.load(GOLDEN)
    mt = int(G[f"isect_{name}__max_tris"])
    s = gpu.preset(name, max_tris=None if mt < 0 else mt)
    with gpu.Context(0, s, gpu.RenderConfig()) as g:
        a = g.intersect_batch(G[f"isect_{name}__org"], G[f"isect_{name}__dir"])
        assert np.array_equal(a["obj"], G[f"isect_{name}__obj"])
        hit = a["obj"] >= 0
        assert rel_err(a["t"][hit], G[f"isect_{name}__t"][hit]).max() <= T_TOL
        assert np.abs(a["nrm"][hit] - G[f"isect_{name}__nrm"][hit]).max() <= T_TOL
        # in fact identical bits except where two coplanar/adjacent triangles tie
        assert (a["t"][hit] == G[f"isect_{name}__t"][hit]).mean() > 0.999
        agree = (a["into"][hit] == G[f"isect_{name}__into"][hit]).mean()
        assert agree > (0.85 if "bump" in name else 0.95), agree  # open height-field: the parity heuristic itself is ~90 % (SURVEY Q8)
        col = g.surface_color(3 if name == "c1_spheres" else 0, G[f"surf_{name}__pos"])
        assert np.array_equal(col, G[f"surf_{name}__col"])


def test_sharded_renderer_on_gpu_engine(gpu, oracle_lib):
    """The host-side render() driver (distributed.py) on the product engine, world 1, against the oracle's render."""
    import torch

    from cgraytracing_b200.distributed import GpuEngine, ShardedRenderer

    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=96, height=64)
    with gpu.Context(0, s, cfg) as g:
        eng = GpuEngine(g, 0)
        img = ShardedRenderer(eng).render(64, 2, 8000)
        # export/import round trip of the hitpoint records leaves the grid unchanged
    with gpu.Context(0, s, cfg) as g2:
        eng2 = GpuEngine(g2, 0)
        g2.eye_pass(32, 64); g2.eye_pass(0, 32)
        rec = eng2.export_hitpoints().clone()
        eng2.import_hitpoints(rec[torch.randperm(rec.shape[0], device=rec.device)])
        r2 = ShardedRenderer(eng2)
        eng2.build_grid()
        r2.round(8000); r2.round(8000)
        img2 = eng2.gather_image(16000.0)
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    for r in range(2):
        o.photon_pass(r * 8000, 8000); o.round_update()
    oimg = o.gather_image(16000.0)
    assert np.allclose(img, oimg, rtol=1e-9, atol=1e-12)
    assert np.allclose(img2, oimg, rtol=1e-9, atol=1e-12)


def test_bezier_surface_statistical_parity(gpu, oracle_lib):
    """Bezier::intersect is a randomised multi-start Newton solve in the reference (bezier.h:233-249); the GPU starts the same
    Newton iteration from a deterministic seed grid. Parity for this primitive is statistical (SURVEY Q14): hit / miss decisions
    and the nearest root must agree on the overwhelming majority of rays, and where both hit, t agrees to 1e-5."""
    s = gpu.preset("c1_spheres_bezier")
    bid = len(s.objects) - 1
    org, dr = camera_rays(1024, 768, 9)
    tgt = np.array([15, -10.1, 35.0]) + np.random.default_rng(5).uniform(-5, 5, (len(org), 3)) * [1, 2, 1]
    dr = tgt - org
    dr /= np.linalg.norm(dr, axis=1)[:, None]
    o = oracle_lib.Oracle(s, gpu.RenderConfig(into_rule=1))
    o.set_libc_rng(1, 1234)
    with gpu.Context(0, s, gpu.RenderConfig()) as g:
        a = g.intersect_batch(org, dr)
    b = o.intersect_batch(org, dr)
    on_a, on_b = a["obj"] == bid, b["obj"] == bid
    assert on_b.sum() > 1000
    assert (on_a == on_b).mean() > 0.97, (on_a == on_b).mean()
    both = on_a & on_b
    close = rel_err(a["t"][both], b["t"][both]) <= T_TOL
    assert close.mean() > 0.97, close.mean()
    # the reference stops Newton at |F| < 1e-6 (bezier.h:26,170): the normal inherits that slack, two seeds of the reference itself
    # agree to ~5e-6; its normal is built from the reference's own dB (not the true Bernstein derivative, bezier.h:37-40)
    dn = np.abs(a["nrm"][both][close] - b["nrm"][both][close]).max(axis=1)
    assert np.median(dn) < 1e-5 and np.quantile(dn, 0.99) < 1e-3, (np.median(dn), np.quantile(dn, 0.99))
    # everything that is not the vase is untouched by the solver: identical
    other = ~on_a & ~on_b
    assert np.array_equal(a["obj"][other], b["obj"][other]) and np.array_equal(a["t"][other], b["t"][other])


def test_full_size_properties_c3(gpu):
    """BASELINE config 3 at its full size (1024x1024, 100,000-triangle glass dragon): size-independent properties.
    sorted keys + consistent cell table; every photon hit accounted for; shard invariance (two GPUs' index ranges == one range);
    accepted-photon counts sum to the deposit counter; one more round only shrinks radii; culling changes no accumulator."""
    s = gpu.preset("c3_dragon_glass")
    cfg = gpu.RenderConfig(width=1024, height=1024)
    N = 1 << 21
    with gpu.Context(0, s, cfg) as g1, gpu.Context(0, s, cfg) as g2:
        for g in (g1, g2):
            g.eye_pass(); g.build_grid()
        hp = g1.download_hitpoints()
        n = len(hp["key"])
        assert n > 1024 * 1024 and g1.counters()["eye_segments"] >= n
        assert np.all(np.diff(hp["key"].astype(np.int64)) >= 0)                       # sorted by bucket key
        same = np.diff(hp["key"].astype(np.int64)) == 0
        assert np.all(np.diff(hp["seq"].astype(np.int64))[same] > 0)                  # creation order inside a bucket
        cs = g1.download_grid().astype(np.int64)
        assert cs[0] == 0 and cs[-1] == n and np.array_equal(np.diff(cs), np.bincount(hp["key"], minlength=cfg.hashsize))
        k, _ = g1.hash_keys(hp["pos"], cfg.hashsize, 200.0 / cfg.height)
        assert np.array_equal(k, hp["key"])                                           # keys are the hash of the stored positions
        # one range vs two disjoint ranges (what two GPUs trace), culling on vs off
        g2.set_culling(False)
        g1.photon_pass(0, N)
        g2.photon_pass(N // 2, N - N // 2); g2.photon_pass(0, N // 2)
        d1, m1 = g1.download_accum(); d2, m2 = g2.download_accum()
        assert np.array_equal(m1, m2)
        assert np.allclose(d1, d2, rtol=1e-9, atol=1e-9)
        c1, c2 = g1.counters(), g2.counters()
        assert c1["deposits"] == c2["deposits"] == int(m1.sum()) > N
        assert c1["photon_segments"] == c2["photon_segments"] and c1["diffuse_hits"] == c2["diffuse_hits"]
        assert c1["photon_segments"] <= 5 * N and c1["diffuse_hits"] <= c1["photon_segments"]
        assert c1["gathered_hits"] <= c1["diffuse_hits"] == c2["gathered_hits"] and c1["candidates"] <= c2["candidates"]
        g1.round_update()
        hp2 = g1.download_hitpoints()
        assert np.array_equal(hp2["n"], m1.astype(np.int32))
        assert np.all(hp2["r2"] <= hp["r2"]) and np.all(hp2["r2"][m1 > 0] < hp["r2"][m1 > 0])
        assert np.all(hp2["flux"] >= 0) and np.isfinite(hp2["flux"]).all()
        img = g1.gather_image(float(N))
        assert np.isfinite(img).all() and img.min() >= 0 and img.mean() > 0.01


@pytest.mark.parametrize("overlap", [0, 1])
def test_chunked_and_pipelined_photon_pass(gpu, oracle_lib, overlap, monkeypatch):
    """A pass split into many chunks (and, with overlap on, pipelined over two streams with double-buffered deposit tables) leaves
    exactly the accumulators of the oracle's single loop."""
    monkeypatch.setenv("CGRT_PHOTON_CHUNK", "7001")
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=128, height=96)
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    with gpu.Context(0, s, cfg) as g:
        g.set_overlap(bool(overlap))
        g.eye_pass(); g.build_grid()
        for r in range(3):
            g.photon_pass(r * 30000, 30000); o.photon_pass(r * 30000, 30000)
            df, m = g.download_accum(); odf, om = o.download_accum()
            assert np.array_equal(m.astype(np.int64), om.astype(np.int64))
            assert np.allclose(df, odf, rtol=1e-9, atol=1e-12)
            g.round_update(); o.round_update()
        assert np.allclose(g.gather_image(90000.0), o.gather_image(90000.0), rtol=1e-9, atol=1e-12)
        assert g.counters()["gpu_launches"] > 3 * 5 * 12


def test_profiled_photon_pass_timing_slots(gpu, monkeypatch):
    """With profiling on, a multi-chunk photon pass over a mesh scene fills every photon-pass slot of timings() (bench.py reports
    them), and the trace slot covers its emission, traversal and continuation parts."""
    monkeypatch.setenv("CGRT_PHOTON_CHUNK", "7001")
    with gpu.Context(0, gpu.preset("c2_bunny_chess"), gpu.RenderConfig(width=128, height=96)) as g:
        g.set_profiling(True)
        g.eye_pass(); g.build_grid()
        g.photon_pass(0, 30000)
        t = g.timings()
    for k in ("photon_trace", "deposit_sort", "photon_deposit", "trace_emit", "trace_traverse", "trace_continue"):
        assert t[k] > 0, (k, t)
    assert t["photon_trace"] >= t["trace_emit"] + t["trace_traverse"] + t["trace_continue"], t


def test_dof_camera_and_samples_bit_exact(gpu, oracle_lib):
    """BASELINE config 4: thin-lens camera (main.cpp:203-207) with num_of_samples > 1 over the displaced floor and the objtype-2 mesh.
    Run twice in one process: the second context re-uses pooled device memory, so anything read before it is written shows up."""
    s = gpu.preset("c4_bump_dof")
    cfg = gpu.RenderConfig(width=160, height=96, use_dof=1, num_of_samples=4, consume_dof_rng=1)
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    b = o.download_hitpoints()
    for attempt in range(2):
        with gpu.Context(0, s, cfg) as g:
            g.eye_pass(); g.build_grid()
            a = g.download_hitpoints()
            assert len(a["pos"]) == len(b["pos"]) > 160 * 96 * 4 * 0.9, (attempt, len(a["pos"]), len(b["pos"]))
            for k in ("key", "hw", "pos", "normal", "f", "r2"):
                assert np.array_equal(a[k], b[k]), (attempt, k)
            assert g.counters()["eye_segments"] == o.counters()["eye_segments"]


def test_eye_pass_small_chunks_and_queue_growth(gpu, oracle_lib, monkeypatch):
    """Many eye-pass chunks with ray queues that have to grow while the wavefront is alive (glass doubles the rays per bounce)."""
    monkeypatch.setenv("CGRT_EYE_CHUNK", "300")
    s = gpu.preset("c2_bunny_chess")
    cfg = gpu.RenderConfig(width=256, height=192)
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    b = o.download_hitpoints()
    with gpu.Context(0, s, cfg) as g:
        g.eye_pass(); g.build_grid()
        a = g.download_hitpoints()
    assert len(a["pos"]) == len(b["pos"]) > 256 * 192
    for k in ("key", "hw", "pos", "normal", "f"):
        assert np.array_equal(a[k], b[k]), k


def test_photon_pass_with_bezier_object(gpu, oracle_lib):
    """BASELINE config 1 (spheres + Bezier vase): the Newton solver is randomised in the reference, so photon-level parity with the
    oracle is statistical: the same photons are traced, a few of the ones that meet the vase resolve differently."""
    s = gpu.preset("c1_spheres_bezier")
    cfg = gpu.RenderConfig(width=128, height=128)
    N = 60000
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass(); o.photon_pass(0, N, o.max_threads())
    with gpu.Context(0, s, cfg) as g:
        g.eye_pass(); g.build_grid()
        assert abs(g.num_hitpoints() - o.num_hitpoints()) <= 0.01 * o.num_hitpoints()
        g.photon_pass(0, N)
        gc, oc = g.counters(), o.counters()
        for k in ("photon_segments", "diffuse_hits", "deposits"):
            assert abs(gc[k] - oc[k]) <= 0.01 * oc[k], (k, gc[k], oc[k])
        g.round_update(); o.round_update()
        a, b = g.gather_image(float(N)), o.gather_image(float(N))
        assert abs(a.mean() - b.mean()) <= 0.01 * b.mean()
        # pixels whose hitpoints are not on the vase see exactly the same photons except those that went through the vase
        assert np.median(np.abs(a - b) / np.maximum(b, 1e-9)) < 1e-3


def test_no_out_of_bounds_writes_with_fenced_buffers():
    """Every scene family, both accumulator modes and the two-stream pipeline with CGRT_GUARD=1: each device buffer sits between two
    4 KiB fences and no kernel may have written into one (stands in for a memory checker, which the GPU pool does not offer)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, CGRT_GUARD="1")
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "sanitize_probe.py")], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "guard mode 1 damaged fence bytes 0" in r.stdout


@pytest.mark.parametrize("hashsize", [97, 4099])
def test_colliding_buckets_are_listed_like_the_reference(gpu, oracle_lib, hashsize):
    """A tiny hash table: many cells share a bucket and several of a photon's 27 neighbour cells hash to the same one, which the reference
    then scans (and deposits into) once per listing (hash.h:35-42, main.cpp:105-122, SURVEY Q13). Counts and fluxes must still equal the
    oracle's, and the GPU must scan exactly the reference's candidates when the reach-map culling is off."""
    W, H, NPH = 64, 48, 12000
    s, cfg, g, o = make(gpu, oracle_lib, "c1_spheres", dict(width=W, height=H, into_rule=1, update_mode=1, hashsize=hashsize), None)
    with g:
        g.set_culling(False)
        g.eye_pass(); g.build_grid()
        o.eye_pass()
        g.photon_pass(0, NPH); o.photon_pass(0, NPH)
        df, m = g.download_accum()
        odf, om = o.download_accum()
        assert np.array_equal(m.astype(np.int64), om.astype(np.int64))
        assert np.allclose(df, odf, rtol=1e-9, atol=1e-12)
        gc, oc = g.counters(), o.counters()
        assert gc["deposits"] == oc["deposits"] and gc["candidates"] == oc["candidates"]
        assert gc["candidates"] > 50 * gc["diffuse_hits"]  # the buckets really are crowded


def test_multisample_image_is_normalised_like_the_reference(gpu, oracle_lib):
    """main.cpp:256 divides by num_photon*num_threads*num_of_samples. Callers state the photons; the samples factor is applied by the
    library (and by the oracle) from the config, so that no entry point can produce a picture num_of_samples times too bright."""
    s = gpu.preset("c4_bump_dof", max_tris=None)
    cfg = gpu.RenderConfig(width=96, height=64, use_dof=1, num_of_samples=4)
    N = 40000
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass(); o.photon_pass(0, N, o.max_threads()); o.round_update()
    with gpu.Context(0, s, cfg) as g:
        g.eye_pass(); g.build_grid(); g.photon_pass(0, N); g.round_update()
        img = g.gather_image(float(N))
        hp = g.download_hitpoints(fields=("flux", "r2", "hw"))
    want = np.zeros_like(img)
    v = hp["flux"] * (1.0 / (3.14159265358979 * hp["r2"] * float(N) * 4.0))[:, None]  # the reference's normaliser, written out
    np.add.at(want, (hp["hw"][:, 0], hp["hw"][:, 1]), v)
    assert img.mean() > 0.01 and np.allclose(img, want, rtol=1e-12, atol=1e-15)
    assert np.allclose(img, o.gather_image(float(N)), rtol=1e-9, atol=1e-12)
