"""The mesh BVH (LBVH build in cgrt_build.cuh, bvh4_closest / root_box_hit in cgrt_device.cuh) against brute force at its edges.

The box tests of the traversal are float arithmetic made conservative by padding (CGRT_BOX_PAD, CGRT_F32_BOUND, the fp64 re-base of far
origins in the F32ONLY instantiation, NaN slabs of zero direction components); they must never decide a hit. Every expected value here
comes from brute force over all triangles (Oracle.mesh_brute) or from the CPU oracle:
  A (CPU)  the oracle's kd-tree equals brute force on every ray set used below, so a GPU-vs-oracle mismatch is the GPU's;
  B        intersect_batch == brute force on degenerate builds (1..5 triangles, equal Morton keys, a zero-extent axis, slivers), trees past
           the float bound, far origins, axis-parallel rays and rays with a component that rounds to zero or a subnormal in float;
  C        the counting instantiations (count_traversal, set_counting) count and change nothing else;
  D        c3 with one triangle past the bound: the fp64-slab eye and photon kernels and the exact root test against the plain scene
           and the oracle (PPM and SPPM);
  E        the F32ONLY re-base of far origins through cgrt_trace, photons and eye rays, against the oracle's trace();
  F        CGRT_TRAV_EXACT (the fp64-slab photon traversal forced on a scene inside the bound) changes no photon.
"""
import functools
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from cgraytracing_b200 import RenderConfig, SceneDesc, preset
from tests.util import assert_flux_close

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FAR_R = (1e2, 1e4, 1e6, 1e8, 1e10)  # at 1e12 the fp64 triangle test itself no longer hits anything: nothing left to miss
FAR_TRI = np.array([[100.0, 100.0, 100.0, 100.1, 100.0, 100.0, 100.0, 100.1, 100.0]])  # behind the ceiling and the right wall of c3


def f32_bound():
    with open(os.path.join(ROOT, "cgraytracing_b200", "csrc", "cgrt_device.cuh")) as fp:
        return float(re.search(r"#define\s+CGRT_F32_BOUND\s+([0-9.eE+-]+)", fp.read()).group(1))


# ---------------------------------------------------------------------------------------------------------------------
# meshes
# ---------------------------------------------------------------------------------------------------------------------
def random_tris(n, seed):
    rng = np.random.default_rng(seed)
    c = rng.uniform(-15, 15, (n, 1, 3))
    return np.ascontiguousarray((c + rng.normal(scale=3.0, size=(n, 3, 3))).reshape(n, 9))


def clustered_tris(seed, n=2000):
    """n small triangles whose centroids lie within 1e-4 of each other (equal Morton keys: the index tie-break of lbvh_delta) and one
    large triangle that stretches the centroid bounds."""
    rng = np.random.default_rng(seed)
    cen = np.array([1.0, 2.0, 3.0]) + rng.uniform(-5e-5, 5e-5, (n, 3))
    a, b = rng.normal(scale=0.1, size=(n, 3)), rng.normal(scale=0.1, size=(n, 3))
    small = np.stack([cen + a, cen + b, cen - a - b], 1).reshape(n, 9)
    return np.concatenate([small, [[-30.0, -20.0, -10.0, 30.0, -20.0, 20.0, 0.0, 30.0, 40.0]]])


def flat_grid(m=24, z=5.0):
    """2 m^2 triangles in the plane z = const: zero centroid extent on one axis."""
    g = np.linspace(-12.0, 12.0, m + 1)
    x0, y0 = np.meshgrid(g[:-1], g[:-1], indexing="ij")
    x1, y1 = np.meshgrid(g[1:], g[1:], indexing="ij")
    x0, y0, x1, y1 = x0.ravel(), y0.ravel(), x1.ravel(), y1.ravel()
    zz = np.full_like(x0, z)
    t1 = np.stack([x0, y0, zz, x1, y0, zz, x0, y1, zz], 1)
    t2 = np.stack([x1, y1, zz, x0, y1, zz, x1, y0, zz], 1)
    return np.ascontiguousarray(np.concatenate([t1, t2]))


def slivers(seed, n=64):
    """Long thin triangles from one face of the box [-20, 20]^3 to the opposite one: every box overlaps every other."""
    rng = np.random.default_rng(seed)
    pa, pb = rng.uniform(-20, 20, (n, 3)), rng.uniform(-20, 20, (n, 3))
    ax = rng.integers(0, 3, n)
    pa[np.arange(n), ax] = -20.0
    pb[np.arange(n), ax] = 20.0
    pc = pb + rng.normal(scale=2e-3, size=(n, 3))
    return np.ascontiguousarray(np.concatenate([pa, pb, pc], 1))


@functools.lru_cache(maxsize=None)
def dragon():
    return preset("c3_dragon_glass", max_tris=20000).objects[-1]["tri9"]


RANDOM_N = (1, 2, 3, 4, 5, 8, 9, 17, 33, 257)
MESHES = [f"random_{n}" for n in RANDOM_N] + ["clustered", "flat_grid", "slivers", "dragon", "dragon_shift", "dragon_x100"]
PAST_BOUND = {"dragon_shift", "dragon_x100"}


@functools.lru_cache(maxsize=None)
def make_mesh(name):
    seed = MESHES.index(name) + 100
    if name.startswith("random_"):
        return random_tris(int(name.split("_")[1]), seed)
    if name == "clustered":
        return clustered_tris(seed)
    if name == "flat_grid":
        return flat_grid()
    if name == "slivers":
        return slivers(seed)
    if name == "dragon":
        return dragon()
    if name == "dragon_shift":
        return np.ascontiguousarray(dragon() + np.tile([1e4, -1e4, 1e4], 3))
    if name == "dragon_x100":
        return np.ascontiguousarray(dragon() * 100.0)
    raise ValueError(name)


def mesh_scene(tri9, col=(0.5, 0.5, 0.5)):
    """The mesh alone, diffuse, no walls: rays can come from any direction."""
    s = SceneDesc(name="mesh_only")
    s.add_mesh(tri9, col, 0.0, 0.0, 1)
    return s


def c3_scene(far):
    """c3 with the dragon cut to 20,000 triangles; far=True appends FAR_TRI to its mesh, which takes the tree past the float bound."""
    s = preset("c3_dragon_glass", max_tris=20000)
    if far:
        s.objects[-1] = dict(s.objects[-1], tri9=np.concatenate([s.objects[-1]["tri9"], FAR_TRI]))
    return s


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2], a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], 1)


def orientation_sign(tri9):
    """Sign of the sum of pa . (pb x pc) in triangle order (orientation_sign in cgrt_api.cu, KDTree::set_orientation in the oracle)."""
    pa, pb, pc = tri9[:, 0:3], tri9[:, 3:6], tri9[:, 6:9]
    c = _cross(pb, pc)
    vol = np.cumsum(pa[:, 0] * c[:, 0] + pa[:, 1] * c[:, 1] + pa[:, 2] * c[:, 2])[-1]  # cumsum: sequential, like the loops
    return 1.0 if vol >= 0.0 else -1.0


def winding_normals(tri9):
    """The raw normal a mesh hit reports: normalize((pa - pb) x (pa - pc)) (objects.h:107) times the mesh's orientation sign, in the same
    fp64 operations."""
    pa, pb, pc = tri9[:, 0:3], tri9[:, 3:6], tri9[:, 6:9]
    n = _cross(pa - pb, pa - pc)
    ln = np.sqrt(n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1] + n[:, 2] * n[:, 2])
    return n * (1 / ln)[:, None] * orientation_sign(tri9)


# ---------------------------------------------------------------------------------------------------------------------
# ray sets
# ---------------------------------------------------------------------------------------------------------------------
def _unit(v):
    return v / np.linalg.norm(v, axis=1)[:, None]


def far_ladder(tri9, rng, per_r):
    """For every R of FAR_R, per_r rays that start at distance R from a vertex (plus 0.05 jitter) and point at it."""
    v = tri9.reshape(-1, 3)
    org, dr = [], []
    for R in FAR_R:
        tgt = v[rng.integers(0, len(v), per_r)] + rng.normal(scale=0.05, size=(per_r, 3))
        o = tgt - _unit(rng.normal(size=(per_r, 3))) * R
        org.append(o)
        dr.append(_unit(tgt - o))
    return np.concatenate(org), np.concatenate(dr)


def ray_sets(tri9, seed, n=2000, per_r=600):
    rng = np.random.default_rng(seed)
    t = tri9.reshape(-1, 3, 3)
    lo, hi = tri9.reshape(-1, 3).min(0), tri9.reshape(-1, 3).max(0)
    c, h = (lo + hi) / 2, np.maximum((hi - lo) / 2, 1.0)
    ar = np.arange(n)

    def inside(m):  # origins in the mesh's box widened by half
        return c + rng.uniform(-1.5, 1.5, (m, 3)) * h

    def centroids(m):
        return t[rng.integers(0, len(t), m)].mean(axis=1)

    out = {}
    out["random"] = (inside(n), _unit(rng.normal(size=(n, 3))))
    k, j = rng.integers(0, len(t), n), rng.integers(0, 3, n)
    tgt = np.where((ar % 2 == 0)[:, None], t[k, j], 0.5 * (t[k, j] + t[k, (j + 1) % 3]))  # vertices, edge midpoints
    o = inside(n)
    out["vertex_edge"] = (o, _unit(tgt - o))
    # axis-parallel: the two other components exactly 0.0 or -0.0
    d = np.where(rng.random((n, 3)) < 0.5, 0.0, -0.0)
    d[ar, rng.integers(0, 3, n)] = rng.choice([-1.0, 1.0], n)
    tgt = centroids(n) + np.where(d == 0, rng.normal(scale=0.02, size=(n, 3)), 0.0)
    out["axis_parallel"] = (tgt - d * (rng.uniform(0.2, 3.0, n) * h.max())[:, None], d)
    # one component 1e-30 (a normal float) or 1e-42 (a float subnormal: its float reciprocal overflows)
    d = _unit(rng.normal(size=(n, 3)))
    ax = rng.integers(0, 3, n)
    d[ar, ax] = 0.0
    d = _unit(d)
    d[ar, ax] = rng.choice([-1.0, 1.0], n) * np.where(ar % 2 == 0, 1e-30, 1e-42)
    out["tiny_component"] = (centroids(n) - d * (rng.uniform(0.2, 3.0, n) * h.max())[:, None], d)
    out["far"] = far_ladder(tri9, rng, per_r)
    return out


def trace_rays(seed):
    """The far-origin rays of E, aimed at the dragon."""
    return far_ladder(dragon(), np.random.default_rng(seed), 400)


PHOTON_SEED, EYE_SEED = 31, 37
# How the deposit kernel's warps happened to group same-cell hits: the order of records inside a counting-sort bin comes from an atomic
# (bin_scatter_kernel), so these two vary from run to run of the same input. Every other counter is a property of the photons.
SCHEDULE_COUNTERS = ("cell_groups", "staged_candidates")


# ---------------------------------------------------------------------------------------------------------------------
# A: the oracle against brute force (CPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mesh", MESHES)
def test_oracle_kd_tree_equals_brute_force(oracle_lib, mesh):
    tri9 = make_mesh(mesh)
    assert (np.abs(tri9).max() > f32_bound()) == (mesh in PAST_BOUND)  # both traversal instantiations are reached below
    o = oracle_lib.Oracle(mesh_scene(tri9), RenderConfig(into_rule=1))
    nrm = winding_normals(tri9)
    for name, (org, d) in ray_sets(tri9, MESHES.index(mesh)).items():
        a = o.intersect_batch(org, d)
        hit, ln, tri = o.mesh_brute(0, org, d)
        hit = hit != 0
        assert np.array_equal(a["obj"] >= 0, hit), (name, int((a["obj"] >= 0).sum()), int(hit.sum()))
        assert np.array_equal(a["t"][hit], ln[hit]), name
        if name != "random":
            assert hit.sum() > 0, name
        same = a["prim"][hit] == tri[hit]
        assert np.array_equal(a["nrm_raw"][hit][same], nrm[tri[hit][same]]), name  # the normal the GPU is held to in B


@pytest.mark.parametrize("seed", [PHOTON_SEED, EYE_SEED])
def test_oracle_kd_tree_equals_brute_force_on_trace_rays(oracle_lib, seed):
    org, d = trace_rays(seed)
    o = oracle_lib.Oracle(mesh_scene(dragon()), RenderConfig(into_rule=1))
    a = o.intersect_batch(org, d)
    hit, ln, _ = o.mesh_brute(0, org, d)
    hit = hit != 0
    assert np.array_equal(a["obj"] >= 0, hit) and hit.mean() > 0.5
    assert np.array_equal(a["t"][hit], ln[hit])


def test_far_triangle_takes_c3_past_the_bound_and_keeps_its_orientation():
    B = f32_bound()
    plain, far = c3_scene(False).objects[-1]["tri9"], c3_scene(True).objects[-1]["tri9"]
    assert np.abs(plain).max() < B - 1.0 and np.abs(far).max() > B
    assert orientation_sign(far) == orientation_sign(plain)


# ---------------------------------------------------------------------------------------------------------------------
# B: intersect_batch against brute force
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mesh", MESHES)
def test_intersect_batch_equals_brute_force(gpu, oracle_lib, mesh):
    """Every ray: the same hit / miss and the same t bits as brute force. Random rays: the same triangle (ties aside, at most 1e-3 of the
    hits) and the same raw normal bits."""
    tri9 = make_mesh(mesh)
    s = mesh_scene(tri9)
    o = oracle_lib.Oracle(s, RenderConfig(into_rule=1))
    nrm = winding_normals(tri9)
    with gpu.Context(0, s, RenderConfig()) as g:
        for name, (org, d) in ray_sets(tri9, MESHES.index(mesh)).items():
            a = g.intersect_batch(org, d)
            hit, ln, tri = o.mesh_brute(0, org, d)
            hit = hit != 0
            gh = a["obj"] >= 0
            assert np.array_equal(gh, hit), (name, int(gh.sum()), int(hit.sum()), np.flatnonzero(gh != hit)[:8])
            assert np.array_equal(a["t"][hit], ln[hit]), (name, np.flatnonzero(a["t"][hit] != ln[hit])[:8])
            if name == "random":
                same = a["prim"][hit] == tri[hit]
                assert (~same).sum() <= 1e-3 * hit.sum(), (int((~same).sum()), int(hit.sum()))
                assert np.array_equal(a["nrm_raw"][hit][same], nrm[tri[hit][same]])


# ---------------------------------------------------------------------------------------------------------------------
# C: counting instantiations
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_count_traversal_of_a_single_triangle(gpu):
    """n = 1: the root is the leaf (no node visit). Rays at its interior test it once each; rays leaving its root box test nothing."""
    tri9 = make_mesh("random_1")
    pa, pb, pc = tri9[0, 0:3], tri9[0, 3:6], tri9[0, 6:9]
    rng = np.random.default_rng(5)
    N = 3000
    u, v = rng.uniform(0.1, 0.45, N), rng.uniform(0.1, 0.45, N)
    p = pa + u[:, None] * (pb - pa) + v[:, None] * (pc - pa)
    nrm = winding_normals(tri9)[0]
    o = p + nrm * rng.uniform(1.0, 20.0, (N, 1)) + rng.normal(scale=0.5, size=(N, 3))
    lo, hi = tri9.reshape(3, 3).min(0), tri9.reshape(3, 3).max(0)
    away_o = np.concatenate([hi + rng.uniform(0.5, 10, (N, 3)), lo - rng.uniform(0.5, 10, (N, 3))])
    away_d = np.concatenate([_unit(rng.uniform(0.05, 1, (N, 3))), -_unit(rng.uniform(0.05, 1, (N, 3)))])
    with gpu.Context(0, mesh_scene(tri9), RenderConfig()) as g:
        assert np.all(g.intersect_batch(o, _unit(p - o))["obj"] == 0)
        assert g.count_traversal(o, _unit(p - o)) == (0, N)
        assert g.count_traversal(away_o, away_d) == (0, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("mesh", ["random_5", "random_257", "clustered", "flat_grid", "dragon", "dragon_shift"])
def test_count_traversal_counts_whole_nodes_and_repeats(gpu, mesh):
    tri9 = make_mesh(mesh)
    sets = ray_sets(tri9, MESHES.index(mesh))
    org = np.concatenate([sets["random"][0], sets["far"][0]])
    d = np.concatenate([sets["random"][1], sets["far"][1]])
    with gpu.Context(0, mesh_scene(tri9), RenderConfig()) as g:
        nv, tt = g.count_traversal(org, d)
        assert g.count_traversal(org, d) == (nv, tt)
        hits = int((g.intersect_batch(org, d)["obj"] >= 0).sum())
    assert nv % 4 == 0 and nv > 0 and tt >= hits > 0, (nv, tt, hits)


@pytest.mark.gpu
def test_counting_photon_pass_changes_only_the_traversal_counters(gpu):
    cfg = RenderConfig(width=64, height=48, into_rule=1, update_mode=1)
    out = []
    for counting in (False, True):
        with gpu.Context(0, c3_scene(False), cfg) as g:
            g.set_counting(counting)
            g.eye_pass(); g.build_grid()
            g.photon_pass(0, 20000)
            out.append(g.download_accum() + (g.counters(),))
    (d0, m0, k0), (d1, m1, k1) = out
    assert np.array_equal(m0, m1) and m0.sum() > 0
    assert np.allclose(d0, d1, rtol=1e-9, atol=1e-12)
    for name in k0:
        if name in ("node_visits", "tri_tests"):
            assert k0[name] == 0 < k1[name], (name, k0[name], k1[name])
        elif name not in SCHEDULE_COUNTERS:
            assert k0[name] == k1[name], (name, k0[name], k1[name])
    assert k1["node_visits"] % 4 == 0


# ---------------------------------------------------------------------------------------------------------------------
# D: the whole pipeline with a tree past the bound
# ---------------------------------------------------------------------------------------------------------------------
def gpu_ctx(gpu, scene, cfg, accum=0):
    g = gpu.Context(0)
    g.set_config(cfg, accum_mode=accum)
    scene.build_into(g)
    g.commit()
    return g


@pytest.mark.gpu
def test_past_bound_eye_pass_equals_plain_scene_and_oracle(gpu, oracle_lib):
    cfg = RenderConfig(width=64, height=48, into_rule=1, update_mode=1)
    with gpu_ctx(gpu, c3_scene(True), cfg) as g, gpu_ctx(gpu, c3_scene(False), cfg) as p:
        for c in (g, p):
            c.eye_pass(); c.build_grid()
        a, b = g.download_hitpoints(), p.download_hitpoints()
        assert g.counters()["eye_segments"] == p.counters()["eye_segments"]
    o = oracle_lib.Oracle(c3_scene(True), cfg)
    o.eye_pass()
    h = o.download_hitpoints()
    assert len(a["pos"]) == len(b["pos"]) == len(h["pos"]) > 0
    for k in ("key", "seq", "hw", "pos", "normal", "f"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("key", "hw", "pos", "normal", "f"):
        assert np.array_equal(a[k], h[k]), k
    assert np.array_equal(a["seq"], (h["path"] * 16 + h["code"]).astype(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
def test_past_bound_photon_rounds_match_oracle(gpu, oracle_lib, accum):
    """Two U2 rounds (radius and flux updated once per round): accepted counts equal to the oracle's and to the plain scene's, flux within
    the accumulator type's bound, segment and deposit counters equal."""
    NPH = 20000
    cfg = RenderConfig(width=64, height=48, into_rule=1, update_mode=1)
    o = oracle_lib.Oracle(c3_scene(True), cfg)
    o.eye_pass()
    th = o.max_threads()
    with gpu_ctx(gpu, c3_scene(True), cfg, accum) as g, gpu_ctx(gpu, c3_scene(False), cfg, accum) as p:
        for c in (g, p):
            c.eye_pass(); c.build_grid()
        for rnd in range(2):
            for c in (g, p):
                c.photon_pass(rnd * NPH, NPH)
            o.photon_pass(rnd * NPH, NPH, th)
            df, m = g.download_accum()
            odf, om = o.download_accum()
            assert np.array_equal(m.astype(np.int64), om.astype(np.int64)) and om.sum() > 0, rnd
            assert np.array_equal(m, p.download_accum()[1]), rnd
            assert_flux_close(df, odf, om, accum)
            for c in (g, p):
                c.round_update()
            o.round_update()
        gc, oc = g.counters(), o.counters()
        for k in ("photon_segments", "diffuse_hits", "deposits"):
            assert gc[k] == oc[k], k


@pytest.mark.gpu
def test_past_bound_sppm_rounds_match_oracle(gpu, oracle_lib):
    """SPPM, jittered camera, two rounds: every round's visible points and accepted counts equal to the oracle's."""
    R, N = 2, 20000
    cfg = RenderConfig(width=64, height=48, into_rule=1, update_mode=1)
    o = oracle_lib.Oracle(c3_scene(True), cfg)
    o.set_sppm(1)
    th = o.max_threads()
    with gpu_ctx(gpu, c3_scene(True), cfg) as g:
        g.set_sppm(1)
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
            om = o.download_accum()[1]
            assert np.array_equal(gm.astype(np.int64), om.astype(np.int64)) and om.sum() > 0, r
            g.round_update()
            o.round_update()


# ---------------------------------------------------------------------------------------------------------------------
# E: the F32ONLY re-base of far origins
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_far_photons_through_trace_deposit_like_the_oracle(gpu, oracle_lib):
    """A diffuse dragon alone (inside the bound: the float-only traversal), photons from the far-origin ladder through cgrt_trace."""
    W, H, FIRST = 64, 48, 4242
    cfg = RenderConfig(width=W, height=H, into_rule=1, update_mode=1)
    s = mesh_scene(dragon(), (0.75, 0.6, 0.5))
    org, d = trace_rays(PHOTON_SEED)
    N = len(org)
    flux = np.tile(np.array([[700.0, 700.0, 700.0]]) * (3.14159265358979 * 4.0), (N, 1))
    with gpu.Context(0, s, cfg) as g:
        g.eye_pass(); g.build_grid()
        g.trace(org, d, flux, False, 0, first_index=FIRST)
        df, m = g.download_accum()
        kg = g.counters()
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    for k in range(N):
        o.trace(org[k], d[k], flux[k], (1, 1, 1), False, path=FIRST + k)
    odf, om = o.download_accum()
    ko = o.counters()
    assert ko["diffuse_hits"] > N // 2
    for k in ("photon_segments", "diffuse_hits", "deposits"):
        assert kg[k] == ko[k], (k, kg[k], ko[k])
    assert om.sum() > 0 and np.array_equal(m.astype(np.int64), om.astype(np.int64))
    assert_flux_close(df, odf, om, 0)


@pytest.mark.gpu
def test_far_eye_rays_through_trace_equal_the_oracle(gpu, oracle_lib):
    """Eye rays from the far-origin ladder, ray i on pixel (i mod W, i div W) so that its path index is i: the hitpoints after build_grid
    equal those the oracle's trace() makes."""
    W, H = 64, 48
    cfg = RenderConfig(width=W, height=H, into_rule=1, update_mode=1)
    s = mesh_scene(dragon(), (0.75, 0.6, 0.5))
    org, d = trace_rays(EYE_SEED)
    N = len(org)
    assert N <= W * H
    x, y = np.arange(N) % W, np.arange(N) // W
    with gpu.Context(0, s, cfg) as g:
        g.trace(org, d, np.ones((N, 3)), True, 0, x, y)
        g.build_grid()
        a = g.download_hitpoints()
        seg = g.counters()["eye_segments"]
    o = oracle_lib.Oracle(s, cfg)
    for i in range(N):
        o.trace(org[i], d[i], (0, 0, 0), (1, 1, 1), True, int(x[i]), int(y[i]), path=i)
    b = o.download_hitpoints()
    assert len(a["pos"]) == len(b["pos"]) > N // 2
    for k in ("key", "hw", "pos", "normal", "f", "r2"):
        assert np.array_equal(a[k], b[k]), k
    assert np.array_equal(a["seq"], (b["path"] * 16 + b["code"]).astype(np.uint32))
    assert seg == o.counters()["eye_segments"]


# ---------------------------------------------------------------------------------------------------------------------
# F: CGRT_TRAV_EXACT
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_forced_exact_traversal_traces_the_same_photons(tmp_path):
    """The library reads CGRT_TRAV_EXACT once per process: the same c3 round in two processes, with and without it."""
    out = []
    for exact in (False, True):
        env = dict(os.environ)
        env.pop("CGRT_TRAV_EXACT", None)
        if exact:
            env["CGRT_TRAV_EXACT"] = "1"
        path = tmp_path / f"exact{int(exact)}.npz"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bvh_exact_worker.py"), str(path)], env=env, capture_output=True, text=True,
                           timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        out.append(np.load(path))
    a, b = out
    assert np.array_equal(a["m"], b["m"]) and a["m"].sum() > 0
    assert np.allclose(a["df"], b["df"], rtol=1e-9, atol=1e-12)
    assert np.array_equal(a["names"], b["names"])
    ka, kb = dict(zip(a["names"].tolist(), a["counters"].tolist())), dict(zip(b["names"].tolist(), b["counters"].tolist()))
    for name in ka:
        if name not in SCHEDULE_COUNTERS:
            assert ka[name] == kb[name], (name, ka[name], kb[name])
    assert ka["photon_segments"] > 0 and ka["deposits"] > 0
