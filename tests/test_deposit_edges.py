"""The deposit kernel's fp32 filters (make_prefilter, prefilter_inner, the cell-box cull and the normal margin in photon_deposit_kernel /
deposit_pair) against a brute-force fp64 gather, on photon-hitpoint pairs placed where those filters can be wrong.

Both sides of every pair are under the test's control: the hitpoints are imported records (cgrt_import_hitpoints_dev /
Oracle.import_hitpoints), the photons are caller-made rays (trace(..., flag=False) with max_depth = 1) that deposit at their first hit and
stop. A ray straight down from (x, -19, z) lands on the floor of walls_only at exactly (x, -20, z); family 3 adds a tilted plane for
photon normals that are not an axis. The brute force restates main.cpp:103-125 in numpy, every fp64 quantity in the reference's
operation order. A numpy float32 emulation of the kernel's filters sorts every pair into the region that decides it (float accept, float
reject, the distance shell or the normal band left to the exact test) and shows, per family, that the filters with a weakened constant
would misdecide some of its pairs:
  1  distance ties (d2 == r2 exactly) and the last / first representable position on either side of r;
  2  coordinates near powers of two whose float roundings move the distance the wrong way by more than E/4, at r (1 +- delta);
  3  hitpoint normals whose dot with the photon normal lies within 1e-6 of EPS, with heavy cancellation (the normal margin);
  4  photons and hitpoints at |x|, |z| up to 1e6 (E grows past r: every pair takes the exact path; the cull box is cells wide);
  5  photons on cell faces and corners, hitpoints across them at r +- ulp, and hitpoints two cells away but within r (gathered only when
     a hash collision lists their bucket);
  6  dense, colliding and straddled cells: 0..300 surviving candidates and 1..600 photons per cell at hashsize 1, 2, 97 and the default.
CPU: brute force == the oracle on every family. GPU: one round in both accumulator modes with the reach map on and off, a second PPM
round at the radii the first round's update left (the pre / pre_n refresh of round_update_kernel), an SPPM round at shrunk pixel radii
(sppm_visible_radius_kernel), and the per-photon update. The peer-memory exchange's copy of the refresh (peer_reduce_update_kernel) needs
two GPUs and is not covered here.
"""
import functools

import numpy as np
import pytest

from cgraytracing_b200 import RenderConfig, preset
from tests.util import assert_flux_close

H, W = 768, 64
R = 200.0 / H                     # main.cpp:84,94
R2 = R * R
CL = 70.0 / np.ceil(70.0 / R)     # hash.h:22-30
LO = np.array([-35.0, -35.0, -15.0])
EPS = 1e-4                        # main.cpp:24
PI = 3.14159265358979             # main.cpp:26
HS = 1000001                      # main.cpp:184
Y0 = -19.0                        # photon origins: t = 1 to the floor
TILT_N = np.array([0.3, 1.0, -0.2]) / np.sqrt(1.09 + 0.04)
F32 = np.float32
OFFS = np.array([(a, b, c) for a in range(3) for b in range(3) for c in range(3)])  # idx outermost, idz innermost (main.cpp:110-112)


def cfg_for(hs, **kw):
    return RenderConfig(width=W, height=H, max_depth=1, hashsize=hs, **kw)


def scene_for(name):
    s = preset("walls_only")
    if name == "tilted":
        s.add_plane((0.0, -10.0, 10.0), TILT_N, (0.6, 0.5, 0.4), 0.0, 0.0)
    return s


# ---------------------------------------------------------------------------------------------------------------------
# grid, brute force, float emulation
# ---------------------------------------------------------------------------------------------------------------------
def cells(p):
    return np.floor((p - LO) / CL).astype(np.int64)  # hash.h:38-42, the IEEE quotient


def buckets(c, hs):
    u = c.astype(np.int32).view(np.uint32)
    v = (u[..., 0] * np.uint32(73856093)) ^ (u[..., 1] * np.uint32(19349663)) ^ (u[..., 2] * np.uint32(83492791))
    return (v % np.uint32(hs)).astype(np.int64)


def candidate_pairs(X, key, hs):
    """-> photon index, hitpoint index and multiplicity of every (photon, hitpoint) pair the 27-bucket gather lists; a bucket listed
    twice among a photon's 27 lists its hitpoints twice."""
    b = buckets(cells(X)[:, None, :] - 1 + OFFS[None], hs)
    u, mult = np.unique(np.arange(len(X))[:, None] * hs + b, return_counts=True)
    p, bb = u // hs, u % hs
    o = np.argsort(key, kind="stable")
    start, end = np.searchsorted(key[o], bb, "left"), np.searchsorted(key[o], bb, "right")
    n = end - start
    first = np.repeat(np.cumsum(n) - n, n)
    hi = o[np.repeat(start, n) + np.arange(n.sum()) - first]
    return np.repeat(p, n), hi, np.repeat(mult, n)


def exact_accept(X, nrm, hp_pos, hp_nrm, r2, pi, hi):
    """main.cpp:116 in the reference's operation order."""
    dd = [hp_pos[hi, a] - X[pi, a] for a in range(3)]
    d2 = dd[0] * dd[0] + dd[1] * dd[1] + dd[2] * dd[2]
    dot = hp_nrm[hi, 0] * nrm[pi, 0] + hp_nrm[hi, 1] * nrm[pi, 1] + hp_nrm[hi, 2] * nrm[pi, 2]
    return (dot > EPS) & (d2 <= r2[hi]), d2, dot


def brute(case, hs, r2=None):
    """-> accepted photons per hitpoint, flux sum per hitpoint (fp64), candidate count, and the pair arrays."""
    hp = case["hp"]
    r2 = np.full(len(hp["pos"]), R2) if r2 is None else r2
    pi, hi, mult = candidate_pairs(case["X"], hp["key"][hs], hs)
    acc, d2, dot = exact_accept(case["X"], case["n"], hp["pos"], hp["nrm"], r2, pi, hi)
    w = np.where(acc, mult, 0)
    n = len(hp["pos"])
    cnt = np.bincount(hi, weights=w, minlength=n).astype(np.int64)
    flux = np.stack([np.bincount(hi, weights=w * ((hp["f"][hi, a] * case["flux"][pi, a]) * (1.0 / PI)), minlength=n) for a in range(3)], 1)
    return dict(cnt=cnt, flux=flux, cand=int(mult.sum()), pi=pi, hi=hi, mult=mult, acc=acc, r2=r2, d2=d2, dot=dot)


def fmaf(a, b, c):
    """fmaf of float32 arrays, rounded once: the fp64 product is exact, and the one case where rounding the fp64 sum again is not the
    single rounding (the sum lands on a float midpoint) is settled by the sign of the sum's error."""
    a, b, c = (np.asarray(x, F32) for x in (a, b, c))
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    s = p + c64
    bb = s - p
    e = (p - (s - bb)) + (c64 - bb)
    f = s.astype(F32)
    f64 = f.astype(np.float64)
    other = np.where(s > f64, np.nextafter(f, F32(np.inf)), np.nextafter(f, F32(-np.inf)))
    tie = (s == (f64 + other.astype(np.float64)) * 0.5) & (e != 0)
    return np.where(tie & ((f64 > s) != (e > 0)), other, f)


def round_dir(x, up):
    f = np.asarray(x).astype(F32)
    if up:
        return np.where(f.astype(np.float64) < x, np.nextafter(f, F32(np.inf)), f)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, F32(-np.inf)), f)


def filter_records(pos, r2, k=4.5e-7):
    """make_prefilter / prefilter_inner: (r + E)^2 rounded up, (r - E)^2 rounded down or -1 when r <= E."""
    r = np.sqrt(r2)
    m = np.maximum(np.maximum(np.abs(pos[:, 0]), np.abs(pos[:, 1])), np.abs(pos[:, 2])) + r + 1.0
    E = k * m
    outer = round_dir((r + E) * (r + E) * (1.0 + 4e-6), True)
    inner = np.where(r <= E, F32(-1.0), round_dir((r - E) * (r - E) * (1.0 - 4e-6), False))
    return outer, inner


def float_decision(case, b, k=4.5e-7, margin=1e-6, shrink=0.0):
    """What the fp32 filters decide for every pair of brute(): 1 accept, 0 reject, -1 left to the exact test; the region (0 float
    accept, 1 float reject, 2 distance shell, 3 normal band); and whether the cell-box cull keeps the pair. k (the constant of E), margin
    (the normal margin's factor; None = no margin at all) and shrink (cull box inset, in cells) emulate weakened filters."""
    hp, pi, hi = case["hp"], b["pi"], b["hi"]
    outer, inner = filter_records(hp["pos"], b["r2"], k)
    q = hp["pos"].astype(F32)[hi]
    qn = hp["nrm"].astype(F32)[hi]
    h = case["X"].astype(F32)[pi]
    hn = case["n"].astype(F32)[pi]
    c = cells(case["X"])[pi]
    b0 = [(LO[a] + c[:, a].astype(np.float64) * CL).astype(F32) for a in range(3)]
    bw = F32(CL)
    bm = F32(1e-5) * (np.abs(b0[0]) + np.abs(b0[1]) + np.abs(b0[2]) + bw + F32(1.0))
    if shrink:
        bm = bm - F32(shrink) * bw
    ex = [np.maximum(np.maximum(b0[a] - bm - q[:, a], q[:, a] - (b0[a] + bw + bm)), F32(0)) for a in range(3)]
    kept = fmaf(ex[2], ex[2], fmaf(ex[1], ex[1], ex[0] * ex[0])) <= outer[hi]
    dd = [q[:, a] - h[:, a] for a in range(3)]
    s = fmaf(dd[2], dd[2], fmaf(dd[1], dd[1], dd[0] * dd[0]))
    dn = fmaf(qn[:, 2], hn[:, 2], fmaf(qn[:, 1], hn[:, 1], qn[:, 0] * hn[:, 0]))
    sn = fmaf(np.abs(qn[:, 2]), np.abs(hn[:, 2]), fmaf(np.abs(qn[:, 1]), np.abs(hn[:, 1]), np.abs(qn[:, 0] * hn[:, 0])))
    mg = np.zeros_like(sn) if margin is None else fmaf(np.full_like(sn, F32(margin)), sn, np.full_like(sn, F32(1e-9)))
    eps = F32(EPS)
    rej = ~kept | (s > outer[hi]) | (dn < eps - mg)
    acc = ~rej & (s <= inner[hi]) & (dn > eps + mg)
    dec = np.where(rej, 0, np.where(acc, 1, -1))
    region = np.where(acc, 0, np.where(rej, 1, np.where(dn > eps + mg, 2, 3)))
    return dec, region, kept


def misdecided(case, b, **kw):
    """Pairs the (weakened) filters decide in fp32 against the reference's outcome."""
    dec = float_decision(case, b, **kw)[0]
    return int(((dec >= 0) & (dec != b["acc"].astype(int))).sum())


# ---------------------------------------------------------------------------------------------------------------------
# placing pairs
# ---------------------------------------------------------------------------------------------------------------------
def d2_of(p, X):
    dx, dy, dz = p[0] - X[0], p[1] - X[1], p[2] - X[2]
    return dx * dx + dy * dy + dz * dz


def ulp_boundary(X, p, axis, r2):
    """Step p[axis] by ulps (away from X = outward) -> (last position with d2 <= r2, first with d2 > r2)."""
    p = np.array(p, dtype=np.float64)
    out = np.inf if p[axis] >= X[axis] else -np.inf
    inw = -out
    while d2_of(p, X) > r2:
        p[axis] = np.nextafter(p[axis], inw)
    while True:
        q = p.copy()
        q[axis] = np.nextafter(p[axis], out)
        if d2_of(q, X) > r2:
            return p, q
        p = q


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.sqrt((v * v).sum(-1, keepdims=True))


def land(scene_name, org, dr):
    """Photon hit points X = o + d t (main.cpp:68, component by component) and face-forwarded normals, from the oracle's intersect."""
    o = _oracle_scene(scene_name)
    hit = o.intersect_batch(org, dr)
    t = hit["t"]
    X = np.stack([org[:, a] + dr[:, a] * t for a in range(3)], 1)
    return X, hit["nrm"].copy(), t


@functools.lru_cache(maxsize=None)
def _oracle_scene(name):
    from oracle import binding as ob

    return ob.Oracle(scene_for(name), cfg_for(HS))


def floor_photons(xz):
    xz = np.asarray(xz, np.float64).reshape(-1, 2)
    org = np.stack([xz[:, 0], np.full(len(xz), Y0), xz[:, 1]], 1)
    return org, np.tile([0.0, -1.0, 0.0], (len(xz), 1))


UP = np.array([0.1, 0.9, -0.2])  # a hitpoint normal the floor normal accepts with a wide margin


class Builder:
    def __init__(self, name, scene, hashsizes, seed):
        self.name, self.scene, self.hashsizes = name, scene, hashsizes
        self.rng = np.random.default_rng(seed)
        self.org, self.dir, self.pos, self.nrm = [], [], [], []

    def photons(self, org, dr):
        X, n, t = land(self.scene, org, dr)
        self.org.append(org)
        self.dir.append(dr)
        return X, n, t

    def hit(self, p, nrm=UP):
        self.pos.append(np.asarray(p, np.float64).reshape(-1, 3))
        self.nrm.append(np.broadcast_to(np.asarray(nrm, np.float64), self.pos[-1].shape).copy())

    def boundary(self, X, dirs, nrm=UP, r2=R2):
        for u in unit(dirs):
            a = int(np.argmax(np.abs(u)))
            pin, pout = ulp_boundary(X, X + np.sqrt(r2) * u, a, r2)
            self.hit([pin, pout], nrm)

    def spread(self, X, k, lo, hi, nrm=UP):
        u = unit(self.rng.normal(size=(k, 3)))
        self.hit(X + R * self.rng.uniform(lo, hi, (k, 1)) * u, nrm)

    def build(self):
        org, dr = np.concatenate(self.org), np.concatenate(self.dir)
        return make_case(self.name, self.scene, org, dr, np.concatenate(self.pos), np.concatenate(self.nrm), self.hashsizes, self.rng)


def make_case(name, scene, org, dr, pos, nrm, hashsizes, rng):
    from oracle import binding as ob

    X, n, t = land(scene, org, dr)
    N = len(pos)
    k0 = ob.hash_keys(pos, HS, R)[0].astype(np.int64)
    order = np.argsort(k0, kind="stable")
    pos, nrm = pos[order], nrm[order]
    hp = dict(pos=pos, nrm=nrm, f=rng.uniform(0.2, 1.0, (N, 3)), key={}, rec={})
    hw = np.stack([np.arange(N) % H, (np.arange(N) // H) % W], 1).astype(np.uint64)
    for hs in hashsizes:
        key = ob.hash_keys(pos, hs, R)[0].astype(np.int64)
        o = np.argsort(key, kind="stable")
        hp["key"][hs] = key
        hp["rec"][hs] = records(pos, nrm, hp["f"], key, hw, o)
    return dict(name=name, scene=scene, org=org, dir=dr, t=t, X=X, n=n, flux=rng.uniform(0.5, 2.0, (len(org), 3)), hp=hp,
                hashsizes=tuple(hashsizes))


def records(pos, nrm, f, key, hw, order):
    """12-double exchange records (include/cgrt.h) in the order `order`; the sort key's low word is the index in canonical order, so the
    canonical order of every hashsize is ascending key, ties in the order of `pos`."""
    n = len(pos)
    seq = np.empty(n, np.uint64)
    seq[order] = np.arange(n, dtype=np.uint64)
    rec = np.zeros((n, 12))
    rec[:, 0:3], rec[:, 3:6], rec[:, 6:9] = pos, nrm, f
    rec[:, 9] = ((key.astype(np.uint64) << np.uint64(32)) | seq).view(np.float64)
    rec[:, 10] = ((hw[:, 0] << np.uint64(32)) | hw[:, 1]).view(np.float64)
    return rec


def canonical(case, hs):
    """The family's hitpoints in the canonical order of hashsize hs (ascending key, ties in the family's order): the order of
    download_accum / download_hitpoints on both sides."""
    return np.argsort(case["hp"]["key"][hs], kind="stable")


# ---------------------------------------------------------------------------------------------------------------------
# the families
# ---------------------------------------------------------------------------------------------------------------------
def fam_ties():
    b = Builder("ties", "floor", (HS,), 1)
    xz = [(0.0, 0.37), (0.0, 7.3), (1.3, 0.0), (-6.1, 0.0), (4.9, 21.7), (-13.3, 9.1), (11.7, 30.3), (-2.9, 15.5)]
    X, _, _ = b.photons(*floor_photons(xz))
    dirs = [(1, 0, 0), (-1, 0, 0), (0, 0, 1), (0, 0, -1), (1, 0, 1), (-1, 0.3, 2), (2, -0.5, -1), (0.2, 1, 0.1), (-0.3, -1, 0.4), (1, 1, 1)]
    for x in X:
        if x[0] == 0.0:   # dd = (r, 0, 0): d2 == r2 exactly
            b.hit([x + (R, 0, 0), x - (R, 0, 0)])
        if x[2] == 0.0:
            b.hit([x + (0, 0, R), x - (0, 0, R)])
        b.boundary(x, dirs)
        b.spread(x, 6, 0.1, 0.9)
        b.spread(x, 6, 1.1, 1.9)
    return b.build()


def fam_rounding():
    """Pairs whose float distance the roundings move by more than E/4 the wrong way, at fp64 distances r (1 +- delta)."""
    rng = np.random.default_rng(2)
    n = 400000
    base = rng.choice([64.0, 128.0, 1024.0, 8192.0], (n, 2)) * rng.choice([-1.0, 1.0], (n, 2))
    X = np.stack([base[:, 0] * (1 + rng.uniform(-2e-3, 4e-3, n)), np.full(n, -20.0), base[:, 1] * (1 + rng.uniform(-2e-3, 4e-3, n))], 1)
    th = rng.uniform(0, 2 * np.pi, n)
    u = unit(np.stack([np.cos(th), rng.uniform(-0.2, 0.2, n), np.sin(th)], 1))
    delta = np.exp(rng.uniform(np.log(1e-9), np.log(1e-5), n)) * rng.choice([-1.0, 1.0], n)
    P = X + (R * (1 + delta))[:, None] * u
    case = dict(X=X, n=np.tile([0.0, 1.0, 0.0], (n, 1)), hp=dict(pos=P, nrm=np.tile(UP, (n, 1))))
    b = dict(pi=np.arange(n), hi=np.arange(n), r2=np.full(n, R2))
    b["acc"] = exact_accept(X, case["n"], P, case["hp"]["nrm"], b["r2"], b["pi"], b["hi"])[0]
    dec4 = float_decision(case, b, k=4.5e-7 / 4)[0]
    wrong = np.flatnonzero((dec4 >= 0) & (dec4 != b["acc"].astype(int)))
    region = float_decision(case, b)[1]
    shell = np.flatnonzero(region == 2)
    keep = np.concatenate([wrong[:160], rng.choice(np.setdiff1d(shell, wrong), 60, replace=False)])
    bl = Builder("rounding", "floor", (HS,), 3)
    bl.photons(*floor_photons(X[keep][:, [0, 2]]))
    bl.hit(P[keep])
    return bl.build()


def fam_normals():
    b = Builder("normals", "tilted", (HS,), 4)
    # the floor normal (0, 1, 0): hn.y == EPS exactly rejects, its upper neighbour accepts
    X, n, _ = b.photons(*floor_photons([(60.0, 0.5), (64.5, -3.0), (70.25, 4.0)]))
    assert np.array_equal(n, np.tile([0.0, 1.0, 0.0], (3, 1)))
    for x in X:
        for hy in (EPS, np.nextafter(EPS, 1.0), np.nextafter(EPS, 0.0), np.nextafter(np.nextafter(EPS, 1.0), 1.0)):
            for a, c in ((0.0, 0.0), (0.8, -0.6), (-0.9, 0.4)):
                b.hit(x + R * 0.3 * unit(b.rng.normal(size=3)), (a, hy, c))
        b.spread(x, 4, 0.1, 0.8, nrm=(0.2, -0.5, 0.1))
    # the tilted plane: hn = (EPS + delta) n + t u, u orthogonal to n, |t| ~ 1 (large components, heavy cancellation)
    xs = np.array([(x, z) for x in (-1.6, -0.4, 0.9, 2.2) for z in (8.3, 10.1, 11.9)])
    org = np.stack([xs[:, 0], np.full(len(xs), 10.0), xs[:, 1]], 1)
    X, n, _ = b.photons(org, np.tile([0.0, -1.0, 0.0], (len(xs), 1)))
    deltas = np.concatenate([np.linspace(-1e-6, 1e-6, 21), np.array([-1, 1]) * 3e-8, np.array([-1, 1]) * 1e-7, np.array([-1, 1]) * 3e-7])
    for x, nn in zip(X, n):
        u1 = unit(np.cross(nn, [0.0, 0.0, 1.0]))
        u2 = np.cross(nn, u1)
        for d in deltas:
            t = b.rng.uniform(0.7, 1.3) * b.rng.choice([-1, 1])
            w = unit(np.cos(b.rng.uniform(0, 6.3)) * u1 + np.sin(b.rng.uniform(0, 6.3)) * u2)
            b.hit(x + R * 0.3 * unit(b.rng.normal(size=3)), (EPS + d) * nn + t * w)
        for _ in range(4):   # ulp steps of one component right at EPS: (last reject, first accept)
            w = unit(np.cos(b.rng.uniform(0, 6.3)) * u1 + np.sin(b.rng.uniform(0, 6.3)) * u2)
            hn = EPS * nn + b.rng.uniform(0.7, 1.3) * w
            a = int(np.argmax(np.abs(nn)))
            step = np.inf if nn[a] > 0 else -np.inf
            dot = lambda v: v[0] * nn[0] + v[1] * nn[1] + v[2] * nn[2]  # noqa: E731
            while dot(hn) > EPS:
                hn[a] = np.nextafter(hn[a], -step)
            while True:
                h2 = hn.copy()
                h2[a] = np.nextafter(hn[a], step)
                if dot(h2) > EPS:
                    break
                hn = h2
            for v in (hn, h2):
                b.hit(x + R * 0.3 * unit(b.rng.normal(size=3)), v)
        b.hit(x + R * 0.2 * unit(b.rng.normal(size=(3, 3))), nn)     # clear accept
        b.hit(x + R * 0.2 * unit(b.rng.normal(size=(3, 3))), -nn)    # clear reject
    return b.build()


def fam_far():
    b = Builder("far", "floor", (HS,), 5)
    xz = []
    for s in (1e2, 1e4, 5e5, 1e6):
        for sx, sz in ((1, 1), (-1, 1), (1, -1), (-1, -1)):
            xz.append((sx * s * 1.03, sz * s * 0.97))
    X, _, _ = b.photons(*floor_photons(xz))
    dirs = [(1, 0, 0), (-1, 0, 0), (0, 0, 1), (1, 0, -1), (-1, 0.2, 1), (0.3, 1, 0.2)]
    for x in X:
        b.boundary(x, dirs)
        b.spread(x, 6, 0.05, 0.95)
        b.spread(x, 6, 1.05, 2.5)
    return b.build()


def face_hashsize():
    """A hashsize under which the bucket of a hitpoint two cells away (in x) collides with one of the photon's 27."""
    c = cells(np.array([[FACE_X + 1e-5, -20.0, FACE_Z + 0.5 * CL]]))[0]
    far = c + np.array([-2, 0, 0])
    for hs in range(101, 100000, 2):
        near = buckets(c - 1 + OFFS, hs)
        if buckets(far[None], hs)[0] in set(near.tolist()):
            return hs
    raise AssertionError("no colliding hashsize")


FACE_K = 134                      # -35 + 134 cl ~ -0.13: the cull box margin bm is smallest near x = z = 0 on the floor
FACE_X = -35.0 + FACE_K * CL
FACE_Z = -15.0 + 58 * CL


def fam_faces():
    hc = face_hashsize()
    b = Builder("faces", "floor", (HS, hc), 6)
    xs = [FACE_X, np.nextafter(FACE_X, -1.0), np.nextafter(FACE_X, 1.0), -35.0 + (FACE_K + 1) * CL, -35.0 + (FACE_K - 1) * CL]
    zs = [FACE_Z, np.nextafter(FACE_Z, 1.0), FACE_Z + 0.5 * CL]
    xz = [(x, z) for x in xs for z in zs]
    X, _, _ = b.photons(*floor_photons(xz))
    dirs = [(1, 0, 0), (-1, 0, 0), (0, 0, 1), (0, 0, -1), (1, 0, 1), (-1, 0, -1), (1, 0, -1), (-1, 0, 1), (-1, 0.5, -1)]
    for x in X:
        b.boundary(x, dirs)
        b.spread(x, 4, 0.5, 1.5)
    # two cells away but within r: the photon just inside its cell's low x face, the hitpoint at 0.9999 r below it
    X2, _, _ = b.photons(*floor_photons([(FACE_X + 1e-5, FACE_Z + 0.5 * CL)]))
    x = X2[0]
    b.hit([x - (0.9999 * R, 0, 0), x - (0.9995 * R, 0, 0), x + (0.9999 * R, 0, 0)])
    return b.build()


DENSE_CAND = (0, 1, 31, 32, 33, 63, 64, 65, 97, 300)
DENSE_PHOT = (1, 31, 32, 33, 255, 256, 257, 600, 32, 1)


def fam_dense():
    b = Builder("dense", "floor", (1, 2, 97, HS), 7)
    cy = cells(np.array([[0.0, -20.0, 0.0]]))[0, 1]
    orgs = []
    for i, (nc, npht) in enumerate(zip(DENSE_CAND, DENSE_PHOT)):
        c = np.array([100 + 3 * i, cy, 50 + (i % 3)])
        lo = LO + c * CL
        if nc:
            p = lo + b.rng.uniform(0.02, 0.98, (nc, 3)) * CL
            nrm = unit(b.rng.normal(size=(nc, 3)) + [0.0, 1.2, 0.0])
            b.hit(p, nrm)
        xz = lo[[0, 2]] + b.rng.uniform(0.01, 0.99, (npht, 2)) * CL
        orgs.append(xz)
    xz = np.concatenate(orgs)
    xz = xz[b.rng.permutation(len(xz))]   # cells interleaved in photon order
    b.photons(*floor_photons(xz))
    return b.build()


FAMILIES = dict(ties=fam_ties, rounding=fam_rounding, normals=fam_normals, far=fam_far, faces=fam_faces, dense=fam_dense)


@functools.lru_cache(maxsize=None)
def family(name):
    from oracle import binding as ob

    ob.build()
    return FAMILIES[name]()


# How many of each family's candidate pairs (with multiplicity, at its first hashsize) each region decides: float accept, float reject,
# distance shell, normal band. The filters weakened as in PINS (E / 4, no normal margin, the cull box 0.1 % of a cell smaller on every
# side) misdecide some pairs of the family named; the shipped filters misdecide none.
REGIONS = dict(ties=(48, 41, 168, 0), rounding=(67, 76, 220, 0), normals=(105, 116, 0, 319), far=(49, 24, 265, 0),
               faces=(1319, 1600, 840, 0), dense=(1974888, 25771041, 27, 0))
PINS = dict(rounding=dict(k=4.5e-7 / 4), normals=dict(margin=None), faces=dict(shrink=1e-3))


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def oracle_round(case, hs):
    from oracle import binding as ob

    o = ob.Oracle(scene_for(case["scene"]), cfg_for(hs))
    o.import_hitpoints(case["hp"]["rec"][hs])
    return o


def oracle_trace(o, case):
    for k in range(len(case["org"])):
        o.trace(case["org"][k], case["dir"][k], case["flux"][k], (0, 0, 0), False, path=k)


@pytest.mark.parametrize("name", list(FAMILIES))
def test_brute_force_equals_oracle(name):
    from oracle import binding as ob

    case = family(name)
    hp = case["hp"]
    assert ob.grid_params(HS, R)[1] == CL
    if case["scene"] == "floor":
        assert np.array_equal(case["t"], np.ones(len(case["t"]))) and np.all(case["X"][:, 1] == -20.0)
    for hs in case["hashsizes"]:
        assert np.array_equal(hp["key"][hs], buckets(cells(hp["pos"]), hs))
        o = oracle_round(case, hs)
        oracle_trace(o, case)
        odf, om = o.download_accum()
        ctr = o.counters()
        b = brute(case, hs)
        o_ = canonical(case, hs)
        assert np.array_equal(om, b["cnt"][o_]), (hs, int(np.abs(om - b["cnt"][o_]).sum()))
        assert ctr["deposits"] == b["cnt"].sum() and ctr["diffuse_hits"] == len(case["org"])
        assert ctr["candidates"] == b["cand"]
        assert np.all(np.abs(odf - b["flux"][o_]) <= 1e-12 * np.abs(b["flux"][o_]))
        assert b["cnt"].sum() > 0 and (b["cnt"] == 0).sum() > 0
    b = brute(case, case["hashsizes"][0])
    region = float_decision(case, b)[1]
    got = np.bincount(region, weights=b["mult"], minlength=4).astype(int)
    assert tuple(got.tolist()) == REGIONS[name], (name, got.tolist())
    if name in PINS:
        assert misdecided(case, b) == 0
        assert misdecided(case, b, **PINS[name]) > 0, name


def test_exact_ties_are_placed():
    """Pairs exactly on both boundaries: d2 == r2 (accepted, `<=` is inclusive) and a normal product == EPS (rejected, `>` is strict)."""
    b = brute(family("ties"), HS)
    assert np.any(b["acc"] & (b["d2"] == R2))
    b = brute(family("normals"), HS)
    tie = b["dot"] == EPS
    assert np.any(tie) and not np.any(b["acc"] & tie) and np.any(b["acc"] & (b["dot"] == np.nextafter(EPS, 1.0)))


def test_faces_pin_the_27_bucket_semantics():
    """The hitpoint two cells away lies within r and is gathered only under the colliding hashsize."""
    case = family("faces")
    hs, hc = case["hashsizes"]
    hp = case["hp"]
    X = case["X"][-1]
    i = int(np.flatnonzero(np.all(hp["pos"] == X - (0.9999 * R, 0, 0), 1))[0])
    assert d2_of(hp["pos"][i], X) <= R2 and cells(hp["pos"][i:i + 1])[0, 0] == cells(X[None])[0, 0] - 2
    last = len(case["X"]) - 1
    for h, listed in ((hs, False), (hc, True)):
        b = brute(case, h)
        sel = (b["pi"] == last) & (b["hi"] == i)
        assert sel.any() == listed and b["acc"][sel].all()


def test_dense_surviving_candidates():
    """Family 6 at the default hashsize: the cull leaves exactly DENSE_CAND candidates to the photons of each cell."""
    case = family("dense")
    b = brute(case, HS)
    kept = float_decision(case, b)[2]
    c = cells(case["X"])[:, 0]
    assert np.bincount(c - 100)[::3].tolist() == list(DENSE_PHOT)
    for p in range(len(c)):
        sel = b["pi"] == p
        assert (b["mult"][sel] * kept[sel]).sum() == DENSE_CAND[(c[p] - 100) // 3]


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def gpu_context(gpu, case, hs, accum=0, cull=True, **kw):
    g = gpu.Context(0)
    g.set_config(cfg_for(hs, **kw), accum_mode=accum)
    scene_for(case["scene"]).build_into(g)
    g.commit()
    g.set_culling(cull)
    return g


def import_records(g, rec):
    import torch

    t = torch.from_numpy(np.ascontiguousarray(rec)).cuda()
    torch.cuda.synchronize()
    g.import_hitpoints_dev(t.data_ptr(), len(rec))
    return t


def gpu_trace(g, case, k=None):
    k = slice(None) if k is None else k
    g.trace(case["org"][k], case["dir"][k], case["flux"][k], flag=False, depth=0)


ROUND_CASES = [(n, hs) for n in FAMILIES for hs in (HS,)] + [("faces", "collide"), ("dense", 1), ("dense", 2), ("dense", 97)]


@pytest.mark.gpu
@pytest.mark.parametrize("accum,cull", [(0, True), (0, False), (1, True), (1, False)])
@pytest.mark.parametrize("name,hs", ROUND_CASES)
def test_gpu_round_equals_brute_force(gpu, name, hs, accum, cull):
    case = family(name)
    if hs == "collide":
        hs = case["hashsizes"][1]
    b = brute(case, hs)
    o = canonical(case, hs)
    with gpu_context(gpu, case, hs, accum, cull) as g:
        hit = g.intersect_batch(case["org"], case["dir"])
        assert np.array_equal(hit["t"], case["t"]) and np.array_equal(hit["nrm"], case["n"])
        t = import_records(g, case["hp"]["rec"][hs])
        g.build_grid()
        gpu_trace(g, case)
        df, m = g.download_accum()
        ctr = g.counters()
        hp = g.download_hitpoints(fields=("pos", "key"))
        del t
    assert np.array_equal(hp["pos"], case["hp"]["pos"][o]) and np.array_equal(hp["key"].astype(np.int64), case["hp"]["key"][hs][o])
    assert np.array_equal(m.astype(np.int64), b["cnt"][o]), int(np.abs(m - b["cnt"][o]).sum())
    assert ctr["deposits"] == b["cnt"].sum() and ctr["diffuse_hits"] == len(case["org"])
    if not cull:
        assert ctr["candidates"] == b["cand"]
    if accum == 0:
        assert np.all(np.abs(df - b["flux"][o]) <= 1e-9 * np.abs(b["flux"][o]))
    else:
        float_flux_close(df, b["flux"][o], b["cnt"][o])


def float_flux_close(df, ref, m):
    """Float accumulators against the fp64 sums. Where hundreds of deposits land on one hitpoint (family 6 at hashsize 1 and 2) their
    float sum in arbitrary order drifts by about sqrt(m) ulp, so only the worst-case bound of assert_flux_close applies there."""
    if m.max() <= 64:
        assert_flux_close(df, ref, m, 1)
    else:
        bound = (np.asarray(m, np.float64)[:, None] + 8.0) * 2.0 ** -24 * np.abs(ref) + 1e-6
        assert np.all(np.abs(df - ref) <= bound)


def shrink_case(seed, ms, scene="floor"):
    """Hitpoints on the floor, 3 units apart; hitpoint i receives ms[i] photons at 0.3 r in round 1."""
    rng = np.random.default_rng(seed)
    k = len(ms)
    pos = np.stack([-15.0 + 3.0 * (np.arange(k) % 10) + rng.uniform(-0.5, 0.5, k), np.full(k, -20.0),
                    2.0 + 3.0 * (np.arange(k) // 10) + rng.uniform(-0.5, 0.5, k)], 1)
    xz = []
    for p, mcount in zip(pos, ms):
        for j in range(mcount):
            a = rng.uniform(0, 2 * np.pi)
            xz.append((p[0] + 0.3 * R * np.cos(a), p[2] + 0.3 * R * np.sin(a)))
    org, dr = floor_photons(xz)
    return make_case("shrink", scene, org, dr, pos, np.tile(UP, (k, 1)), (HS,), rng)


def second_round(case, r2):
    """Round-2 photons around every hitpoint at its radius r2: the ulp boundary in several directions and rings between the new radius and
    the old one."""
    rng = np.random.default_rng(11)
    pos = case["hp"]["pos"]
    xz = []
    for p, rr in zip(pos, r2):
        for th in np.linspace(0.0, 2 * np.pi, 7)[:-1] + rng.uniform(0, 1):
            u = np.array([np.cos(th), 0.0, np.sin(th)])
            X0 = p + np.sqrt(rr) * u    # photon X on the floor at distance r from the hitpoint; the boundary in X.x
            a = 0 if abs(u[0]) >= abs(u[2]) else 2
            xin, xout = ulp_boundary(p, X0, a, rr)
            xz += [(xin[0], xin[2]), (xout[0], xout[2])]
        for f in (0.5, 1.0 + 1e-6, 1.0 + 1e-4, 0.5 * (1.0 + np.sqrt(R2 / rr)), np.sqrt(R2 / rr) * (1 - 1e-4)):
            th = rng.uniform(0, 2 * np.pi)
            xz.append((p[0] + f * np.sqrt(rr) * np.cos(th), p[2] + f * np.sqrt(rr) * np.sin(th)))
    org, dr = floor_photons(xz)
    X, n, _ = land("floor", org, dr)
    return dict(case, org=org, dir=dr, X=X, n=n, flux=rng.uniform(0.5, 2.0, (len(org), 3)))


MS = (1, 2, 3, 5, 0, 1, 8, 2, 1, 4, 13, 0, 1, 1, 2, 6, 3, 1, 9, 2)


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
def test_gpu_second_round_at_updated_radii(gpu, accum):
    """round_update shrinks the radii of the hitpoints round 1 reached; round 2 decides at the new radius (pre / pre_n refreshed)."""
    case = shrink_case(21, MS)
    o = oracle_round(case, HS)
    oracle_trace(o, case)
    o.round_update()
    with gpu_context(gpu, case, HS, accum) as g:
        t = import_records(g, case["hp"]["rec"][HS])
        g.build_grid()
        gpu_trace(g, case)
        g.round_update()
        r2 = g.download_hitpoints(fields=("r2",))["r2"]
        assert np.array_equal(r2, o.download_hitpoints(fields=("r2",))["r2"])
        assert np.array_equal(canonical(case, HS), np.arange(len(r2)))  # one hashsize: canonical order is the order of the records
        assert np.sum(r2 < R2) == sum(1 for m in MS if m)
        c2 = second_round(case, r2)
        gpu_trace(g, c2)
        df, m = g.download_accum()
        del t
    oracle_trace(o, c2)
    odf, om = o.download_accum()
    b = brute(c2, HS, r2=r2)
    assert np.array_equal(om, b["cnt"])
    assert np.array_equal(m.astype(np.int64), b["cnt"]), (m.tolist(), b["cnt"].tolist())
    if accum == 0:
        assert np.all(np.abs(df - odf) <= 1e-9 * np.abs(odf))
    else:
        float_flux_close(df, odf, om)
    region = float_decision(c2, b)[1]
    assert np.sum(region == 2) > 0 and np.sum(region == 0) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("accum", [0, 1])
def test_gpu_sppm_round_at_pixel_radii(gpu, accum):
    """SPPM: the crafted visible points take their pixel's radius (sppm_visible_radius_kernel), which round 1 shrank."""
    from oracle import binding as ob

    case = shrink_case(22, MS)
    rec = case["hp"]["rec"][HS]
    o = ob.Oracle(scene_for("floor"), cfg_for(HS))
    o.set_sppm(2)
    with gpu_context(gpu, case, HS, accum) as g:
        g.set_sppm(2)
        for r, c in ((0, case), (1, None)):
            g.sppm_eye_pass(r, 0, 0)
            o.sppm_eye_pass(r, 0, 0)
            t = import_records(g, rec)
            o.import_hitpoints(rec)
            g.build_grid()
            o.build_grid()
            if c is None:
                pix = g.sppm_download_pixels()
                hw = np.stack([np.arange(len(rec)) % H, (np.arange(len(rec)) // H) % W], 1)
                r2 = pix["r2"][hw[:, 0], hw[:, 1]]
                assert np.sum(r2 < R2) == sum(1 for m in MS if m)
                c = second_round(case, r2)
                b = brute(c, HS, r2=r2)
            gpu_trace(g, c)
            oracle_trace(o, c)
            if r == 1:
                _, m = g.download_accum()
                assert np.array_equal(m.astype(np.int64), b["cnt"]), (m.tolist(), b["cnt"].tolist())
            g.round_update()
            o.round_update()
            del t
        pix, opix = g.sppm_download_pixels(), o.sppm_download_pixels()
    assert np.array_equal(pix["n"], opix["n"]) and np.array_equal(pix["r2"], opix["r2"])
    tol = 1e-9 if accum == 0 else 2e-6
    assert np.all(np.abs(pix["tau"] - opix["tau"]) <= tol * np.abs(opix["tau"]) + 1e-300)


def one_photon_per_hitpoint(case):
    """The photons of a boundary family thinned so that no hitpoint is accepted by two of them (the outcome is order-free)."""
    b = brute(case, HS)
    taken, keep = set(), []
    for p in range(len(case["org"])):
        hs_ = set(b["hi"][(b["pi"] == p) & b["acc"]].tolist())
        if not hs_ & taken:
            keep.append(p)
            taken |= hs_
    k = np.array(keep)
    return dict(case, org=case["org"][k], dir=case["dir"][k], X=case["X"][k], n=case["n"][k], flux=case["flux"][k], t=case["t"][k])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ties", "rounding", "normals", "far", "faces"])
def test_gpu_per_photon_update(gpu, name):
    case = one_photon_per_hitpoint(family(name))
    b = brute(case, HS)
    assert b["cnt"].max() == 1
    o = canonical(case, HS)
    with gpu_context(gpu, case, HS, update_mode=0) as g:
        t = import_records(g, case["hp"]["rec"][HS])
        g.build_grid()
        gpu_trace(g, case)
        n = g.download_hitpoints(fields=("n",))["n"]
        del t
    assert np.array_equal(n.astype(np.int64), b["cnt"][o])


@pytest.mark.gpu
@pytest.mark.parametrize("what", ["key_past_hashsize", "key_not_the_cell", "row_outside", "column_outside"])
def test_gpu_import_refuses_bad_records(gpu, what):
    case = family("ties")
    rec = case["hp"]["rec"][HS].copy()
    bad = rec.copy()
    i = len(rec) // 2
    sk = bad[i:i + 1, 9].view(np.uint64)
    hw = bad[i:i + 1, 10].view(np.uint64)
    key = sk >> np.uint64(32)
    low = sk & np.uint64(0xFFFFFFFF)
    if what == "key_past_hashsize":
        sk[:] = (np.uint64(HS) << np.uint64(32)) | low
    elif what == "key_not_the_cell":
        sk[:] = (((key + np.uint64(1)) % np.uint64(HS)) << np.uint64(32)) | low
    elif what == "row_outside":
        hw[:] = (np.uint64(H) << np.uint64(32)) | (hw & np.uint64(0xFFFFFFFF))
    else:
        hw[:] = (hw & ~np.uint64(0xFFFFFFFF)) | np.uint64(W)
    import cgraytracing_b200 as cg

    with gpu_context(gpu, case, HS) as g:
        t = import_records(g, rec)
        assert g.num_hitpoints() == len(rec)
        with pytest.raises(cg.CgrtError, match="import"):
            import_records(g, bad)
        assert g.num_hitpoints() == len(rec)
        g.build_grid()
        gpu_trace(g, case)
        _, m = g.download_accum()
        del t
    assert np.array_equal(m.astype(np.int64), brute(case, HS)["cnt"][canonical(case, HS)])
