"""Which object a ray hits when the choice is close: the closest-hit rule of main.cpp:50-63 against the kernels that split it.

The reference walks the objects in insertion order and keeps a hit only if it is strictly nearer: on an exact tie the object listed first
wins. The kernels split that loop by object class and across kernels (analytic_phase / plane_take, deferred_wanted, deferred_resolve,
closest_hit_block, photon_bezier_kernel, photon_traverse_kernel) and rely on the lexicographic minimum of (len, object index) instead. Ties
almost never happen by chance, so every case here is crafted with exact arithmetic: axis-parallel rays over integer (Pythagorean) geometry.
  A  exact ties between planes, spheres, meshes and a displaced floor, in every order: the CPU proves the ties real and the oracle's pick the
     lowest index; intersect_batch, eye rays and photon rays through cgrt_trace must equal the oracle bit for bit;
  B  an exact copy of an object: listed after it, invisible; listed before it with another colour and material, the original recoloured
     (full PPM and SPPM passes, the GPU against itself);
  C  tangent sphere rays, origins on a surface, rays parallel to a plane: intersect_batch and eye rays against the oracle;
  D  textures on x-, y-, z-normal and tilted planes: texel boundaries, rims, the texteps band; surface_color and eye hitpoints;
  E  the table limits: a full scene commits and resolves its ties; one more object, texture, Bezier surface or tree is refused;
  F  a Bezier surface's top cap against a plane at the same height, both orders, with the GPU as its own reference.
"""
import functools
import itertools

import numpy as np
import pytest

from cgraytracing_b200 import CgrtError, RenderConfig, SceneDesc, preset
from tests.util import assert_flux_close

FAR_TRI = np.array([[100.0, 100.0, 100.0, 100.1, 100.0, 100.0, 100.0, 100.1, 100.0]])  # takes the scene's trees past CGRT_F32_BOUND
FLUX0 = np.array([700.0, 700.0, 700.0]) * (3.14159265358979 * 4.0)
MIRROR = 0.8
# How the deposit kernel's warps grouped same-cell hits (an atomic orders records inside a counting-sort bin), and the traversal work
SCHEDULE_COUNTERS = ("cell_groups", "staged_candidates")
TRAVERSAL_COUNTERS = ("node_visits", "tri_tests", "exact_tests")


# ---------------------------------------------------------------------------------------------------------------------
# A: crafted exact ties
# ---------------------------------------------------------------------------------------------------------------------
# A sphere of radius R centred at (0, 0, Z0), and a plane, a two-triangle mesh and a displaced floor in y = b. A ray parallel to y at
# horizontal distance a from the centre, with a^2 + b^2 = R^2, meets the sphere exactly where it meets y = b: l.l - tca^2 = a^2 and
# sqrt(R^2 - a^2) = b, all in integers. Down rays start at y = b + 8 (len 8, the t0 branch); up rays start inside the sphere at y = -3
# (len b + 3, the t1 branch).
Z0 = 20.0
GEOMS = {
    "down13": dict(R=13.0, b=12.0, y0=20.0, dy=-1.0, legs=[(3, 4), (5, 0)]),
    "down25": dict(R=25.0, b=20.0, y0=28.0, dy=-1.0, legs=[(9, 12), (15, 0)]),
    "up25": dict(R=25.0, b=15.0, y0=-3.0, dy=1.0, legs=[(12, 16), (20, 0)]),
}
# partners of a family: P plane (normal +y), P2 the same plane given by another point and the opposite normal, S sphere, S2 its copy,
# M mesh, M2 its copy, D displaced floor (a bump texture whose grid texels are black: its triangles lie exactly in the flat plane)
FAMILIES = {
    "down13": ("down13", ("P", "S", "M", "D")),
    "down25": ("down25", ("P", "S", "M", "D")),
    "up25": ("up25", ("P", "S", "M", "D")),
    "planes": ("down13", ("P", "P2", "S", "M")),
    "meshes": ("down13", ("M", "M2", "P", "S")),
    "spheres": ("up25", ("S", "S2", "P", "D")),
}
CLASS = dict(P="plane", P2="plane", S="sphere", S2="sphere", M="mesh", M2="mesh", D="floor")
COLOURS = dict(P=(0.9, 0.3, 0.2), P2=(0.2, 0.8, 0.3), S=(0.3, 0.4, 0.9), S2=(0.7, 0.7, 0.2), M=(0.6, 0.2, 0.7), M2=(0.2, 0.6, 0.6),
               D=(0.5, 0.5, 0.5))
BUMP_W = 66  # lenx = W, leny = H: grid vertex j sits at p.x + 3 j exactly


def tie_rays(geom):
    g = GEOMS[geom]
    offs = set()
    for p, q in g["legs"]:
        for sp in (1, -1):
            for sq in (1, -1):
                offs.add((sp * p, sq * q))
                offs.add((sq * q, sp * p))
    offs = sorted(offs)
    org = np.array([[float(x), g["y0"], Z0 + z] for x, z in offs])
    d = np.tile([0.0, g["dy"], 0.0], (len(org), 1))
    return org, d


def tie_len(geom):
    g = GEOMS[geom]
    return abs(g["b"] - g["y0"])


@functools.lru_cache(maxsize=None)
def bump_rgb():
    """Grid texels (rows and columns that are multiples of 3) black, so height 1 - exp(0) = 0; every other texel coloured."""
    rgb = np.zeros((BUMP_W, BUMP_W, 3), np.uint8)
    rgb[..., 0], rgb[..., 1], rgb[..., 2] = 150, 170, 190
    rgb[::3, ::3] = 0
    return rgb


def quad(b, half=30.0):
    """Two triangles in y = b over |x|, |z - Z0| <= half. Their shared edge runs along x = -(z - Z0), which no tie ray meets."""
    a, c, e, f = (-half, b, Z0 - half), (half, b, Z0 - half), (-half, b, Z0 + half), (half, b, Z0 + half)
    return np.array([a + c + e, f + e + c], dtype=np.float64)


def add_partner(s, role, geom, col, refl, tex):
    g = GEOMS[geom]
    if role == "P":
        s.add_plane((0.0, g["b"], 0.0), (0, 1, 0), col, refl)
    elif role == "P2":
        s.add_plane((5.0, g["b"], -7.0), (0, -1, 0), col, refl)
    elif role in ("S", "S2"):
        s.add_sphere((0.0, 0.0, Z0), g["R"], col, refl)
    elif role in ("M", "M2"):
        s.add_mesh(quad(g["b"]), col, refl)
    elif role == "D":
        s.add_plane((0.0, g["b"], 0.0), (0, 1, 0), col, refl, 0.0, tex)
    else:
        raise ValueError(role)


def tie_scene(family, order, extra=0, diffuse=None, catchers=False, far=False):
    """The partners of `family` in `order` (a permutation of its roles). extra: dummy planes listed first, far off and parallel to every tie
    ray (nplane mod 3 of the three-at-a-time plane loop). diffuse: the one diffuse role, the others mirrors (None: all diffuse). catchers:
    diffuse planes at y = +-60 that take what the mirrors send up or down. far: a last mesh with FAR_TRI."""
    geom, _ = FAMILIES[family]
    s = SceneDesc(name=f"ties_{family}")
    tex = s.add_texture(bump_rgb(), (0, 1, 0), (-31.5, 0.0, Z0 - 31.5), BUMP_W, BUMP_W, True) if "D" in order else -1
    for k in range(extra):
        s.add_plane((500.0 + 10 * k, 0.0, 0.0), (-1, 0, 0), (0.4, 0.4, 0.4))
    for role in order:
        refl = 0.0 if diffuse is None or role == diffuse else MIRROR
        add_partner(s, role, geom, COLOURS[role], refl, tex)
    if catchers:
        s.add_plane((0.0, 60.0, 0.0), (0, -1, 0), (0.8, 0.8, 0.8))
        s.add_plane((0.0, -60.0, 0.0), (0, 1, 0), (0.6, 0.6, 0.6))
    if far:
        s.add_mesh(FAR_TRI, (0.5, 0.5, 0.5))
    return s


PERMS = list(itertools.permutations(range(4)))


def orders_of(family, perms=PERMS):
    roles = FAMILIES[family][1]
    return [tuple(roles[i] for i in p) for p in perms]


def trace_orders(family):
    """Every rotation of the partner list and its reverse: each partner comes first once and meets every other one in both orders."""
    roles = FAMILIES[family][1]
    rots = [roles[k:] + roles[:k] for k in range(4)]
    return rots + [tuple(reversed(r)) for r in rots]


def cfg_small(max_depth=5):
    return RenderConfig(width=32, height=24, into_rule=1, update_mode=1, max_depth=max_depth)


# --- CPU ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("family", list(FAMILIES))
def test_ties_are_exact_and_the_oracle_picks_the_first(oracle_lib, family):
    geom, roles = FAMILIES[family]
    org, d = tie_rays(geom)
    L = tie_len(geom)
    winners = set()
    for order in orders_of(family):
        o = oracle_lib.Oracle(tie_scene(family, order), RenderConfig(into_rule=1))
        lens = []
        for k, role in enumerate(order):
            hit, ln, _ = o.object_intersect(k, org, d)
            assert np.all(hit == 1), (order, role)
            lens.append(ln)
            if role == "D":  # the displaced triangles tie with the flat plane too: the reference keeps the plane (lenp < len is strict)
                th, tl, _ = o.mesh_brute(k, org, d)
                assert np.all(th != 0) and np.all(tl == L), order
        lens = np.array(lens)
        assert np.all(lens == L), (order, lens)  # every partner, every ray: the same len bit for bit, so every class pair ties
        a = o.intersect_batch(org, d)
        assert np.all(a["obj"] == 0) and np.all(a["t"] == L), order
        if order[0] == "D":
            assert np.all(a["prim"] == -1) and np.all(a["nrm_raw"] == [0.0, 1.0, 0.0])
        winners.add(order[0])
    assert winners == set(roles)  # the winner's class changes with the order: a kernel that ignores the order fails somewhere
    assert {CLASS[r] for r in winners} == {CLASS[r] for r in roles}


@pytest.mark.parametrize("geom", ["down13", "up25"])
def test_displaced_floor_is_coloured_at_every_tie_point(oracle_lib, geom):
    """Black texels only under the grid vertices: a diffuse displaced floor never has f = 0 at a tie point (flux / max(f) stays finite)."""
    org, d = tie_rays(geom)
    s = tie_scene("down13" if geom == "down13" else "spheres", ("D",))
    o = oracle_lib.Oracle(s, RenderConfig(into_rule=1))
    X = org + d * tie_len(geom)
    assert np.all(o.surface_color(0, X).max(axis=1) > 0)


# --- GPU: intersect_batch ---------------------------------------------------------------------------------------------
def assert_hits_equal(a, b, what):
    assert np.array_equal(a["obj"], b["obj"]), (what, a["obj"], b["obj"])
    for k in ("t", "nrm", "nrm_raw", "prim"):
        assert np.array_equal(a[k], b[k]), (what, k)


@pytest.mark.gpu
@pytest.mark.parametrize("family", list(FAMILIES))
def test_intersect_batch_breaks_ties_like_the_oracle(gpu, oracle_lib, family):
    """Every order of the four partners; 0, 1 or 2 dummy planes in front, so that the plane loop ends with each remainder mod 3."""
    geom, _ = FAMILIES[family]
    org, d = tie_rays(geom)
    for n, order in enumerate(orders_of(family)):
        extra = n % 3
        s = tie_scene(family, order, extra=extra)
        with gpu.Context(0, s, RenderConfig()) as g:
            a = g.intersect_batch(org, d)
        b = oracle_lib.Oracle(s, RenderConfig(into_rule=1)).intersect_batch(org, d)
        assert np.all(b["obj"] == extra)  # the first partner: the dummy planes come before it
        assert_hits_equal(a, b, order)


# --- GPU: eye rays and photons through cgrt_trace ------------------------------------------------------------------------
def compare_eye_hitpoints(g, o, what, allow_empty=False):
    """-> the number of hitpoints (allow_empty: a mirror inside a mirror sphere can keep every path off the diffuse surfaces)."""
    a, b = g.download_hitpoints(), o.download_hitpoints()
    assert len(a["pos"]) == len(b["pos"]) > (-1 if allow_empty else 0), what
    for k in ("key", "hw", "pos", "normal", "f", "r2"):
        assert np.array_equal(a[k], b[k]), (what, k)
    assert np.array_equal(a["seq"], (b["path"] * 16 + b["code"]).astype(np.uint32)), what
    return len(b["pos"])


def eye_trace_both(g, o, org, d, W):
    N = len(org)
    x, y = np.arange(N) % W, np.arange(N) // W
    g.trace(org, d, np.ones((N, 3)), True, 0, x, y)
    for i in range(N):
        o.trace(org[i], d[i], (0, 0, 0), (1, 1, 1), True, int(x[i]), int(y[i]), path=i)


@pytest.mark.gpu
@pytest.mark.parametrize("far", [False, True])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_tied_eye_rays_through_trace_equal_the_oracle(gpu, oracle_lib, family, far):
    """eye_bounce_kernel's closest_hit_block<F32> (far: the fp64-slab instantiation): one diffuse partner, mirrors of distinct colours, so
    the f of a hitpoint (on the partner or on a catcher) tells which partner won."""
    geom, roles = FAMILIES[family]
    org, d = tie_rays(geom)
    cfg = cfg_small()
    nhp = 0
    for n, order in enumerate(trace_orders(family)):
        s = tie_scene(family, order, extra=n % 3, diffuse=roles[n % 4], catchers=True, far=far)
        o = oracle_lib.Oracle(s, cfg)
        with gpu.Context(0, s, cfg) as g:
            eye_trace_both(g, o, org, d, cfg.width)
            g.build_grid()
            nhp += compare_eye_hitpoints(g, o, order, allow_empty=True)
            assert g.counters()["eye_segments"] == o.counters()["eye_segments"], order
    assert nhp > 0


@pytest.mark.gpu
@pytest.mark.parametrize("max_depth", [1, 2])
@pytest.mark.parametrize("far", [False, True])
@pytest.mark.parametrize("family", list(FAMILIES))
def test_tied_photons_through_trace_deposit_like_the_oracle(gpu, oracle_lib, family, far, max_depth):
    """photon_inject_kernel, photon_traverse_kernel<F32> (far: F32 = false) and the continuation kernel. The eye rays along the tie rays
    put hitpoints where the diffuse partner wins; photons along the same rays (eight paths each) deposit there when it wins for them too."""
    geom, roles = FAMILIES[family]
    org0, d0 = tie_rays(geom)
    org, d = np.repeat(org0, 8, axis=0), np.repeat(d0, 8, axis=0)
    N, FIRST = len(org), 777
    cfg = cfg_small(max_depth)
    flux = np.tile(FLUX0, (N, 1))
    for n, order in enumerate(trace_orders(family)):
        s = tie_scene(family, order, extra=n % 3, diffuse=roles[n % 4], catchers=True, far=far)
        o = oracle_lib.Oracle(s, cfg)
        with gpu.Context(0, s, cfg) as g:
            eye_trace_both(g, o, org0, d0, cfg.width)
            g.build_grid()
            g.trace(org, d, flux, False, 0, first_index=FIRST)
            df, m = g.download_accum()
            kg = g.counters()
        for k in range(N):
            o.trace(org[k], d[k], flux[k], (1, 1, 1), False, path=FIRST + k)
        odf, om = o.download_accum()
        ko = o.counters()
        for k in ("photon_segments", "diffuse_hits", "deposits"):
            assert kg[k] == ko[k], (order, k, kg[k], ko[k])
        assert np.array_equal(m.astype(np.int64), om.astype(np.int64)), order
        assert_flux_close(df, odf, om, 0)
        if order[0] == roles[n % 4]:
            assert ko["diffuse_hits"] >= N and om.sum() > 0, order  # the diffuse partner won: every photon's first segment ends on it


# ---------------------------------------------------------------------------------------------------------------------
# B: duplicate objects on full passes
# ---------------------------------------------------------------------------------------------------------------------
def with_copy(base, src, where, **over):
    """base with a copy of object `src` inserted at index `where` (over: fields changed in the copy)."""
    s = SceneDesc(name=base.name, textures=list(base.textures), objects=list(base.objects))
    s.objects.insert(where, dict(s.objects[src], **over))
    return s


def recoloured(base, src, **over):
    s = SceneDesc(name=base.name, textures=list(base.textures), objects=list(base.objects))
    s.objects[src] = dict(s.objects[src], **over)
    return s


def c3_far():
    s = preset("c3_dragon_glass", max_tris=20000)
    s.objects[-1] = dict(s.objects[-1], tri9=np.concatenate([s.objects[-1]["tri9"], FAR_TRI]))
    return s


DUP_CASES = {
    # name: (base scene, object copied, fields of the coloured copy)
    "c1_sphere": (lambda: preset("c1_spheres"), 2, dict(col=np.array([0.2, 0.9, 0.4]), refl=0.0, transp=0.0)),
    "c3_dragon": (lambda: preset("c3_dragon_glass", max_tris=20000), 5, dict(col=np.array([0.75, 0.6, 0.5]), refl=0.0, transp=0.0)),
    "c3_dragon_far": (c3_far, 5, dict(col=np.array([0.75, 0.6, 0.5]), refl=0.0, transp=0.0)),
    "bump_floor": (lambda: preset("default_bump"), 0, dict(col=np.array([0.9, 0.9, 0.9]), refl=MIRROR)),
    "c1_vase": (lambda: preset("c1_spheres_bezier"), 8, dict(col=np.array([0.4, 0.7, 0.9]), refl=0.0)),
}


def full_round(gpu, scene, sppm, nph):
    cfg = RenderConfig(width=48, height=36, into_rule=1, update_mode=1)
    with gpu.Context(0, scene, cfg) as g:
        if sppm:
            g.set_sppm(1)
            g.sppm_begin_round(0)
        else:
            g.eye_pass()
            g.build_grid()
        hp = g.download_hitpoints(fields=("pos", "normal", "f", "key", "seq", "hw", "r2"))
        g.photon_pass(0, nph)
        df, m = g.download_accum()
        return hp, df, m, g.counters()


def assert_same_round(x, y, what):
    (ha, dfa, ma, ka), (hb, dfb, mb, kb) = x, y
    assert len(ha["pos"]) == len(hb["pos"]) > 0, what
    for k in ha:
        assert np.array_equal(ha[k], hb[k]), (what, k)
    assert np.array_equal(ma, mb) and mb.sum() > 0, what
    assert_flux_close(dfa, dfb, mb, 0)
    for k in ka:
        # gpu_launches: the copy's tree is built by launches of its own
        if k not in SCHEDULE_COUNTERS + TRAVERSAL_COUNTERS + ("gpu_launches",):
            assert ka[k] == kb[k], (what, k, ka[k], kb[k])


@pytest.mark.gpu
@pytest.mark.parametrize("sppm", [0, 1])
@pytest.mark.parametrize("case", list(DUP_CASES))
def test_copied_object_after_is_invisible_and_before_recolours(gpu, case, sppm):
    """PPM eye pass (eye_bounce_kernel<true, F32>) or one SPPM jitter round, then one emission round of 1 Mi photons."""
    make, src, over = DUP_CASES[case]
    base = make()
    nph = 1 << 20
    ref = full_round(gpu, base, sppm, nph)
    assert_same_round(full_round(gpu, with_copy(base, src, src + 1), sppm, nph), ref, (case, "after"))
    ref2 = full_round(gpu, recoloured(base, src, **over), sppm, nph)
    assert_same_round(full_round(gpu, with_copy(base, src, src, **over), sppm, nph), ref2, (case, "before"))


# ---------------------------------------------------------------------------------------------------------------------
# C: tangent, on-surface and parallel rays
# ---------------------------------------------------------------------------------------------------------------------
TAN_SPHERES = [((3.0, 0.0, 30.0), 7.0), ((3.0, 0.0, 60.0), 7.3), ((3.0, 0.0, 90.0), 10.0), ((3.0, 0.0, 120.0), 0.5)]


def tangent_scene():
    s = SceneDesc(name="tangent")
    for c, r in TAN_SPHERES:
        s.add_sphere(c, r, (0.7, 0.5, 0.3))
    s.add_plane((200.0, 0.0, 0.0), (-1, 0, 0), (0.4, 0.6, 0.8))  # backstop: a ray that grazes past still ends somewhere
    return s


def tangent_rays():
    """Along +x at height y = r (d2 == r2 exactly when the sums are exact) and its ulp neighbours, from a near and a far origin."""
    org = []
    for (cx, cy, cz), r in TAN_SPHERES:
        ys = [r]
        for k in (1, 2, 3, 5, 8, 13, 40, 200):
            ys += [np.nextafter(r, np.inf) if k == 1 else r + k * np.spacing(r), r - k * np.spacing(r)]
            ys += [r * (1 + k * 2.0 ** -45), r * (1 - k * 2.0 ** -45)]
        for dist in (2 * r, 60.0):
            for y in ys:
                org.append((cx - dist, cy + y, cz))
                org.append((cx - dist, cy - y, cz))
    org = np.array(org)
    return org, np.tile([1.0, 0.0, 0.0], (len(org), 1))


def surface_scene():
    s = SceneDesc(name="surfaces")
    s.add_sphere((0.0, 0.0, 30.0), 9.5, (0.8, 0.3, 0.3))
    s.add_plane((0.0, -12.0, 0.0), (0, 1, 0), (0.3, 0.8, 0.3))
    s.add_plane((0.0, 0.0, 55.0), (0, 0, -1), (0.3, 0.3, 0.8))
    s.add_plane((31.0, 0.0, 0.0), (-1, 0, 0), (0.6, 0.6, 0.2))
    return s


def _unit(v):
    return v / np.linalg.norm(v, axis=1)[:, None]


def on_surface_rays(oracle_lib, seed=3, n=1500):
    """Origins on the sphere or a plane, made as a bounce makes them (X = o + d t of a previous hit), leaving outward and inward."""
    rng = np.random.default_rng(seed)
    s = surface_scene()
    o = oracle_lib.Oracle(s, RenderConfig(into_rule=1))
    org0 = np.column_stack([rng.uniform(-25, 25, n), rng.uniform(-10, 20, n), rng.uniform(0, 20, n)])
    tgt = np.where((np.arange(n) % 2 == 0)[:, None], np.array([0.0, 0.0, 30.0]) + rng.normal(scale=6.0, size=(n, 3)),
                   np.column_stack([rng.uniform(-30, 30, n), np.full(n, -12.0), rng.uniform(0, 50, n)]))
    d0 = _unit(tgt - org0)
    a = o.intersect_batch(org0, d0)
    hit = a["obj"] >= 0
    X = org0[hit] + d0[hit] * a["t"][hit][:, None]
    nrm = a["nrm"][hit]  # face-forwarded: points back to where the ray came from
    dr = _unit(rng.normal(size=(len(X), 3)))
    side = np.sign(np.sum(dr * nrm, axis=1))
    out = dr * side[:, None]
    return np.concatenate([X, X]), np.concatenate([out, -out]), a["obj"][hit]


def parallel_rays(seed=5, n=400):
    """Directions in the plane y = const (y component +0.0 or -0.0), from above, below and on the floor y = -12."""
    rng = np.random.default_rng(seed)
    d = _unit(np.column_stack([rng.normal(size=n), np.zeros(n), rng.normal(size=n)]))
    d[:, 1] = np.where(np.arange(n) % 2 == 0, 0.0, -0.0)
    y = np.choose(np.arange(n) % 3, [np.full(n, -12.0), rng.uniform(-11.9, 10, n), rng.uniform(-30, -12.1, n)])
    org = np.column_stack([rng.uniform(-20, 20, n), y, rng.uniform(0, 50, n)])
    return org, d


def test_tangent_family_has_hits_and_misses(oracle_lib):
    o = oracle_lib.Oracle(tangent_scene(), RenderConfig(into_rule=1))
    org, d = tangent_rays()
    per = len(org) // len(TAN_SPHERES)
    for k in range(len(TAN_SPHERES)):
        hit, _, _ = o.object_intersect(k, org[k * per:(k + 1) * per], d[k * per:(k + 1) * per])
        assert 0 < hit.sum() < per, (k, int(hit.sum()), per)


def test_on_surface_origins_reach_the_zero_numerator(oracle_lib):
    """Some bounce origins on the floor give (p - X).n == 0 exactly (plane_len's shortcut), others a few ulp; both sides of the sphere."""
    X, dr, obj = on_surface_rays(oracle_lib)
    fl = np.concatenate([obj, obj]) == 1
    num = (0.0 - X[:, 0]) * 0.0 + (-12.0 - X[:, 1]) * 1.0 + (0.0 - X[:, 2]) * 0.0
    assert (num[fl] == 0.0).sum() > 0 and (num[fl] != 0.0).sum() > 0
    sp = np.concatenate([obj, obj]) == 0
    assert sp.sum() > 100 and fl.sum() > 100


def c_sets(oracle_lib):
    X, dr, _ = on_surface_rays(oracle_lib)
    return {"tangent": (tangent_scene(),) + tangent_rays(), "on_surface": (surface_scene(), X, dr),
            "parallel": (surface_scene(),) + parallel_rays()}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["tangent", "on_surface", "parallel"])
def test_grazing_rays_equal_the_oracle(gpu, oracle_lib, name):
    s, org, d = c_sets(oracle_lib)[name]
    b = oracle_lib.Oracle(s, RenderConfig(into_rule=1)).intersect_batch(org, d)
    with gpu.Context(0, s, RenderConfig()) as g:
        a = g.intersect_batch(org, d)
    assert_hits_equal(a, b, name)
    cfg = RenderConfig(width=64, height=64, into_rule=1, update_mode=1)
    assert len(org) <= cfg.width * cfg.height
    o = oracle_lib.Oracle(s, cfg)
    with gpu.Context(0, s, cfg) as g:
        eye_trace_both(g, o, org, d, cfg.width)
        g.build_grid()
        compare_eye_hitpoints(g, o, name)


# ---------------------------------------------------------------------------------------------------------------------
# D: textures on every plane orientation
# ---------------------------------------------------------------------------------------------------------------------
TEX_W, TEX_H = 5, 7
TILT = np.array([-0.6, 0.8, 0.0])
TILT_T = np.array([0.8, 0.6, 0.0])  # in the tilted plane


@functools.lru_cache(maxsize=None)
def tex_rgb():
    """5 wide, 7 high, every texel its own colour."""
    i, j = np.meshgrid(np.arange(TEX_H), np.arange(TEX_W), indexing="ij")
    return np.stack([10 + 35 * i, 10 + 45 * j, np.full_like(i, 100)], -1).astype(np.uint8)


# (plane point, plane normal, texture normal, texture origin, lenx, leny); the room's walls at +-20, floor and ceiling at +-20, back at 40
TEX_PLANES = {
    "x": ((-20.0, 0.0, 0.0), (1, 0, 0), (1.0, 0.0, 0.0), (-20.0, -17.0, 3.0), 10.5, 23.75),
    "y": ((0.0, -20.0, 0.0), (0, 1, 0), (0.0, 1.0, 0.0), (-21.0, -20.0, -5.0), 42.0, 45.5),
    "z": ((0.0, 0.0, 40.0), (0, 0, -1), (0.0, 0.0, 1.0), (-20.0, -20.0, 40.0), 40.0, 37.5),
    "tilt": ((-12.0, -20.0, 0.0), tuple(TILT), tuple(TILT), (-12.0, -20.0, 0.0), 9.0, 30.0),
}


def texture_scene():
    s = SceneDesc(name="textures")
    for k, (p, n, tn, tp, lx, ly) in enumerate(TEX_PLANES.values()):
        t = s.add_texture(tex_rgb(), tn, tp, lx, ly, False)
        s.add_plane(p, n, (0.2 + 0.1 * k, 0.3, 0.4), 0.0, 0.0, t)
    s.add_plane((20.0, 0.0, 0.0), (-1, 0, 0), (0.15, 0.5, 0.15))
    s.add_plane((0.0, 20.0, 0.0), (0, -1, 0), (0.5, 0.5, 0.5))
    return s


def edge_values(L, n):
    """Texel boundaries k L / n and the rims, each with ulp neighbours, the texteps band near 0, and two interior points."""
    v = []
    for k in range(n + 1):
        b = k * L / n
        v += [b, np.nextafter(b, np.inf), np.nextafter(np.nextafter(b, np.inf), np.inf), np.nextafter(b, -np.inf),
              np.nextafter(np.nextafter(b, -np.inf), -np.inf)]
    v += [0.005, 0.0099, 0.0101, 0.37 * L, 0.81 * L, L - 0.005]
    return np.array(sorted(set(v)))


def texture_points(name):
    p, n, tn, tp, lx, ly = TEX_PLANES[name]
    tp = np.array(tp)
    if name == "x":   # branch 1: dd.y over lenx (rows, H), dd.z over leny (columns, W)
        u, v = edge_values(lx, TEX_H), edge_values(ly, TEX_W)
        U, V = np.meshgrid(u, v, indexing="ij")
        return np.column_stack([np.full(U.size, tp[0]), tp[1] + U.ravel(), tp[2] + V.ravel()])
    if name == "y":   # branch 2: dd.x over lenx (columns, W), dd.z over leny (rows, H); |dd.x| < texteps falls into branch 1
        u, v = edge_values(lx, TEX_W), edge_values(ly, TEX_H)
        U, V = np.meshgrid(u, v, indexing="ij")
        return np.column_stack([tp[0] + U.ravel(), np.full(U.size, tp[1]), tp[2] + V.ravel()])
    if name == "z":   # branch 3: dd.x over lenx (columns, W), dd.y over leny (rows, flipped)
        u, v = edge_values(lx, TEX_W), edge_values(ly, TEX_H)
        U, V = np.meshgrid(u, v, indexing="ij")
        return np.column_stack([tp[0] + U.ravel(), tp[1] + V.ravel(), np.full(U.size, tp[2])])
    # tilted: s along TILT_T, w along z; the bands |dd.x| < 0.01 (|s| < 0.0125) and |dd.y| < 0.01 (|s| < 0.0167)
    s = np.array([-0.02, -0.0167, -0.0166, -0.0126, -0.0124, -0.005, -1e-4, 0.0, 1e-4, 0.005, 0.0124, 0.0126, 0.0166, 0.0167, 0.02, 1.0, 5.0, -3.0])
    w = np.concatenate([edge_values(ly, TEX_H), [-1.0, ly + 1.0]])
    S, Wv = np.meshgrid(s, w, indexing="ij")
    return tp + S.ravel()[:, None] * TILT_T + Wv.ravel()[:, None] * np.array([0.0, 0.0, 1.0])


def texture_branch(name, pts):
    """Which branch of Texture::color a point takes (0, 1, 2: the x, y, z band; 3: none) and its unclamped (row, column): numpy replays the
    fp64 operations in the reference's order."""
    _, _, tn, tp, lx, ly = TEX_PLANES[name]
    tn, tp = np.array(tn), np.array(tp)
    dd = pts - tp
    dot = dd[:, 0] * tn[0] + dd[:, 1] * tn[1] + dd[:, 2] * tn[2]
    dd = dd - tn[None, :] * dot[:, None]
    eps = 1e-2
    bx, by, bz = np.abs(dd[:, 0]) < eps, np.abs(dd[:, 1]) < eps, np.abs(dd[:, 2]) < eps
    br = np.where(bx, 0, np.where(by, 1, np.where(bz, 2, 3)))
    with np.errstate(invalid="ignore"):
        r = np.select([br == 0, br == 1, br == 2], [np.floor(dd[:, 1] / lx * TEX_H), np.floor(dd[:, 2] / ly * TEX_H),
                                                    TEX_H - 1 - np.floor(dd[:, 1] / ly * TEX_H)], -1)
        c = np.select([br == 0, br == 1, br == 2], [np.floor(dd[:, 2] / ly * TEX_W), np.floor(dd[:, 0] / lx * TEX_W),
                                                    np.floor(dd[:, 0] / lx * TEX_W)], -1)
    return br, r.astype(int), c.astype(int)


OWN_BRANCH = {"x": 0, "y": 1, "z": 2}


@pytest.mark.parametrize("name", list(TEX_PLANES))
def test_texture_samples_reach_every_branch_and_rim(oracle_lib, name):
    o = oracle_lib.Oracle(texture_scene(), RenderConfig(into_rule=1))
    tid = list(TEX_PLANES).index(name)
    pts = texture_points(name)
    hit, col, rc = o.texture_color(tid, pts)
    br, r, c = texture_branch(name, pts)
    h = hit == 1
    # the oracle's texel is the replayed one: the clamp never changes an index. Division of a value below the rim by the rim rounds to at
    # most 1 - 2^-53, and that times W or H to below W or H, so no sampled point (boundaries, rims, their ulp neighbours) reaches the clamp.
    assert np.array_equal(rc[h, 0], r[h]) and np.array_equal(rc[h, 1], c[h])
    assert np.all((r[h] >= 0) & (r[h] < TEX_H) & (c[h] >= 0) & (c[h] < TEX_W))
    if name in OWN_BRANCH:
        b = OWN_BRANCH[name]
        assert np.all(br[h] == b) and h.sum() > 50
        assert len(set(zip(r[h], c[h]))) == TEX_W * TEX_H  # every texel, so a flipped or swapped index shows in the colour
        assert (~h).sum() > 0  # the rims 0, lenx, leny are outside (strict <)
        if name == "y":
            assert np.any(br == 0)  # |dd.x| < texteps sends a floor point to the first branch, which reports no texel
            assert not np.any(h & (br == 0))
    else:
        assert np.any(h & (br == 0)) and np.any(h & (br == 1)) and np.any(br == 3) and not np.any(h & (br == 3))
    assert np.array_equal(col[h], tex_rgb()[r[h], c[h]] / 256.0)


@pytest.mark.gpu
def test_surface_color_on_every_orientation_equals_the_oracle(gpu, oracle_lib):
    s = texture_scene()
    o = oracle_lib.Oracle(s, RenderConfig(into_rule=1))
    with gpu.Context(0, s, RenderConfig()) as g:
        for k, name in enumerate(TEX_PLANES):
            pts = texture_points(name)
            assert np.array_equal(g.surface_color(k, pts), o.surface_color(k, pts)), name


@pytest.mark.gpu
def test_textured_walls_eye_pass_equals_the_oracle(gpu, oracle_lib):
    cfg = RenderConfig(width=96, height=72, into_rule=1, update_mode=1)
    s = texture_scene()
    o = oracle_lib.Oracle(s, cfg)
    o.eye_pass()
    with gpu.Context(0, s, cfg) as g:
        g.eye_pass()
        g.build_grid()
        a = g.download_hitpoints()
    b = o.download_hitpoints()
    assert len(a["pos"]) == len(b["pos"]) > 0
    for k in ("key", "hw", "pos", "normal", "f"):
        assert np.array_equal(a[k], b[k]), k
    assert len({tuple(f) for f in b["f"]}) > TEX_W * TEX_H // 2  # many texels are seen


# ---------------------------------------------------------------------------------------------------------------------
# E: table limits
# ---------------------------------------------------------------------------------------------------------------------
VASE_CP = [(0, -10, 4), (0, 2, 4), (0, -2, 0), (0, 10, 2)]
CAP = dict(OBJECTS=12, BVH=4, TEX=4, BEZIER=2)


def full_table_scene(order):
    """12 objects, 4 trees (M, D, M2 and a far-off mesh), 2 Bezier surfaces and 4 textures; the down13 partners in `order` among them.
    The vases and the dummy planes lie where no tie ray reaches their boxes, so the oracle draws no random numbers."""
    s = tie_scene("down13", order)
    for k in range(3):
        t = s.add_texture(tex_rgb(), (1, 0, 0), (500.0 + 10 * k, 0, 0), 5, 5, False)
        s.add_plane((500.0 + 10 * k, 0.0, 0.0), (-1, 0, 0), (0.4, 0.4, 0.4), 0.0, 0.0, t)
    s.add_mesh(quad(GEOMS["down13"]["b"]), COLOURS["M2"])
    s.add_mesh(FAR_TRI + np.tile([-300.0, 0.0, 0.0], 3), (0.5, 0.5, 0.5))
    s.add_bezier(VASE_CP, (300.0, 0.0, 0.0), (0.9, 0.9, 0.9))
    s.add_bezier(VASE_CP, (-300.0, 0.0, 0.0), (0.9, 0.9, 0.9))
    s.add_plane((0.0, 0.0, 900.0), (0, 0, -1), (0.4, 0.4, 0.4))
    assert len(s.objects) == CAP["OBJECTS"] and len(s.textures) == CAP["TEX"]
    return s


def refused(gpu, scene, at_commit):
    g = gpu.Context(0)
    try:
        g.set_config(RenderConfig())
        with pytest.raises(CgrtError) as e:
            scene.build_into(g)
            assert at_commit, "the scene was taken whole"
            g.commit()
        assert "status -4" in str(e.value), str(e.value)
    finally:
        g.close()


@pytest.mark.gpu
def test_full_tables_commit_and_resolve_ties(gpu, oracle_lib):
    org, d = tie_rays("down13")
    for order in orders_of("down13", PERMS[::5]):
        s = full_table_scene(order)
        with gpu.Context(0, s, RenderConfig()) as g:
            a = g.intersect_batch(org, d)
        b = oracle_lib.Oracle(s, RenderConfig(into_rule=1)).intersect_batch(org, d)
        assert np.all(b["obj"] == 0)
        assert_hits_equal(a, b, order)


@pytest.mark.gpu
def test_one_more_entry_is_refused(gpu):
    full = full_table_scene(("P", "S", "M", "D"))
    s = SceneDesc(name="objects", textures=list(full.textures), objects=full.objects + [dict(full.objects[0])])
    refused(gpu, s, at_commit=False)  # cgrt_add_plane
    s = SceneDesc(name="textures", textures=full.textures + [full.textures[1]], objects=[])
    refused(gpu, s, at_commit=False)  # cgrt_add_texture
    s = SceneDesc(name="bezier")
    for k in range(CAP["BEZIER"] + 1):
        s.add_bezier(VASE_CP, (30.0 * k, 0.0, 0.0), (0.9, 0.9, 0.9))
    refused(gpu, s, at_commit=True)
    s = SceneDesc(name="trees")
    for k in range(CAP["BVH"] + 1):
        s.add_mesh(quad(float(k)), (0.5, 0.5, 0.5))
    refused(gpu, s, at_commit=True)


# ---------------------------------------------------------------------------------------------------------------------
# F: a Bezier surface against a later plane
# ---------------------------------------------------------------------------------------------------------------------
VASE_POS = (15.0, -10.1, 35.0)


def vase_box_top():
    """Z.box[2] of cgrt_commit_scene: the largest control-point y plus pos.y, in fp64."""
    return max(float(p[1]) for p in VASE_CP) + VASE_POS[1]


def cap_rays(seed=11, n=4000):
    """From outside the vase's wall, 0.1 and more below its rim, up through the cap disc (radius |cp[-1].z| = 2): the wall gives Newton a
    root, and the cap then overrides len with (box[2] - o.y) / d.y."""
    rng = np.random.default_rng(seed)
    top = vase_box_top()
    phi, rho = rng.uniform(0, 2 * np.pi, n), rng.uniform(4.5, 12.0, n)
    org = np.column_stack([VASE_POS[0] + rho * np.cos(phi), rng.uniform(-19.0, -3.0, n), VASE_POS[2] + rho * np.sin(phi)])
    psi, r2 = rng.uniform(0, 2 * np.pi, n), rng.uniform(0, 1.9, n)
    tgt = np.column_stack([VASE_POS[0] + r2 * np.cos(psi), np.full(n, top), VASE_POS[2] + r2 * np.sin(psi)])
    return org, _unit(tgt - org)


def vase_plane_scene(order, vase_refl=0.0, plane_refl=0.0, normal=(0, 1, 0), catcher=False):
    s = SceneDesc(name="vase_plane")
    for k in order:
        if k == "V":
            s.add_bezier(VASE_CP, VASE_POS, (0.9, 0.5, 0.2), vase_refl)
        else:
            s.add_plane((0.0, vase_box_top(), 0.0), normal, (0.2, 0.5, 0.9), plane_refl)
    if catcher:
        s.add_plane((0.0, -60.0, 0.0), (0, 1, 0), (0.6, 0.6, 0.6))
    return s


@functools.lru_cache(maxsize=None)
def _cap_tie_rays(gpu):
    org, d = cap_rays()
    with gpu.Context(0, vase_plane_scene("V"), RenderConfig()) as g:
        v = g.intersect_batch(org, d)
    with gpu.Context(0, vase_plane_scene("P"), RenderConfig()) as g:
        p = g.intersect_batch(org, d)
    keep = (v["obj"] == 0) & (p["obj"] == 0) & (v["t"] == p["t"])
    assert np.all(v["nrm_raw"][keep] == [0.0, 1.0, 0.0])  # the cap's normal: the tie is the cap's, not the wall's
    return org[keep], d[keep], p["t"][keep]


@pytest.mark.gpu
def test_vase_cap_ties_a_plane_at_its_box_top(gpu):
    org, d, t = _cap_tie_rays(gpu)
    assert len(org) >= 100, len(org)


@pytest.mark.gpu
@pytest.mark.parametrize("normal", [(0, 1, 0), (0, -1, 0)])
def test_vase_and_plane_tie_goes_to_the_first(gpu, normal):
    """closest_hit_block's Bezier branch through intersect_batch and eye rays (f shows the winner)."""
    org, d, t = _cap_tie_rays(gpu)
    N = len(org)
    cfg = RenderConfig(width=64, height=64, into_rule=1, update_mode=1, max_depth=1)
    assert N <= cfg.width * cfg.height
    for order in ("VP", "PV"):
        s = vase_plane_scene(order, normal=normal)
        col = np.array(s.objects[0]["col"])
        with gpu.Context(0, s, RenderConfig()) as g:
            a = g.intersect_batch(org, d)
        assert np.all(a["obj"] == 0) and np.array_equal(a["t"], t), order
        with gpu.Context(0, s, cfg) as g:
            g.trace(org, d, np.ones((N, 3)), True, 0, np.arange(N) % cfg.width, np.arange(N) // cfg.width)
            g.build_grid()
            h = g.download_hitpoints()
        assert len(h["f"]) == N and np.all(h["f"] == col), order


@pytest.mark.gpu
@pytest.mark.parametrize("diffuse", ["V", "P"])
def test_vase_and_plane_tie_for_photons_goes_to_the_first(gpu, diffuse):
    """photon_bezier_kernel merges the vase into the plane's hit: one of the two diffuse, the other a mirror, one segment per photon. The
    photon's first hit is diffuse exactly when the diffuse object is listed first."""
    org, d, t = _cap_tie_rays(gpu)
    N = len(org)
    cfg = RenderConfig(width=64, height=64, into_rule=1, update_mode=1, max_depth=1)
    # eye rays straight down below the plane, onto the catcher: the grid is never empty
    eo = np.column_stack([np.linspace(-40, -30, 16), np.full(16, -30.0), np.full(16, 5.0)])
    ed = np.tile([0.0, -1.0, 0.0], (16, 1))
    for order in ("VP", "PV"):
        s = vase_plane_scene(order, vase_refl=0.0 if diffuse == "V" else MIRROR, plane_refl=0.0 if diffuse == "P" else MIRROR, catcher=True)
        with gpu.Context(0, s, cfg) as g:
            g.trace(eo, ed, np.ones((16, 3)), True, 0, np.arange(16), np.zeros(16, np.int32))
            g.build_grid()
            g.trace(org, d, np.tile(FLUX0, (N, 1)), False, 0, first_index=99)
            k = g.counters()
        assert k["photon_segments"] == N, order
        assert k["diffuse_hits"] == (N if order[0] == diffuse else 0), (order, k["diffuse_hits"], N)
