"""CPU: the comparisons of tests/test_oracle_vs_ref.py and the live mirror test of tests/test_mirror.py, against stored outputs so that
they run without the compiled reference: tests/golden/ref_live.npz, written by tests/golden/make_golden_live.py.

Each case below runs the same inputs through either side: "ref" (the compiled reference, oracle/_ref/libcgref.so, where present) or
"oracle" (oracle/ppm_oracle.hpp). The fixture keeps, per case, a SHA-256 digest of the inputs and of every output array (bit-exact
comparison of the whole output) plus a seeded sample of the output rows (what differs, when a digest does not match). Its `source`
names the side that wrote it; `test_stored_outputs_equal_the_live_reference` checks the stored outputs against the reference itself
wherever the reference is built."""
import hashlib
import os
import tempfile

import numpy as np
import pytest

from cgraytracing_b200 import RenderConfig, preset
from tests.util import camera_rays

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_live.npz")
SAMPLE_ROWS = 200
REF_W, REF_H = 1024, 768  # the reference's compiled-in image size (main.cpp)
HP_FIELDS = ("pos", "normal", "f", "flux", "r2", "n", "hw", "key")  # what the reference's hitpoint download returns


def digest(arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


def _bezier(ob, side):
    """Bezier::intersect's randomised Newton solve (bezier.h:233-249) drawing from the same rand() stream on both sides."""
    s = preset("c1_spheres_bezier")
    bid = len(s.objects) - 1
    org, dr = camera_rays(1024, 768, 29)
    # aim half of the rays at the vase so that Newton actually runs
    tgt = np.array([15, -10.1, 35.0]) + np.random.default_rng(5).uniform(-5, 5, (len(org) // 2, 3)) * [1, 2, 1]
    d2 = tgt - org[: len(tgt)]
    d2 /= np.linalg.norm(d2, axis=1)[:, None]
    dr[: len(tgt)] = d2
    if side == "ref":
        e = ob.Ref(s)
        e.seed(99)
    else:
        e = ob.Oracle(s, RenderConfig(into_rule=0))
        e.set_libc_rng(1, 99)
    h, ln, nrm = e.object_intersect(bid, org, dr)
    hit = h > 0
    assert hit.sum() > 100
    return [org, dr], {"hit": h, "t": np.where(hit, ln, 0.0), "nrm": np.where(hit[:, None], nrm, 0.0)}


MESH_TEXTS = {
    0: "begin\nvertex 0 0 0\nvertex 1 0 0.5\nvertex 0 1 -2\nend\n\nbegin\nvertex 1 1 1\nvertex 2 1 1\nvertex 1 3 1.25\nend\n\n",
    1: "4\nv  0 0 0\nv  1 0 0\nv  0 1 0\nv  0 0 1\n2\nf 1 2 3 \nf 1 3 4 \n",
}


def _mesh_loader(ob, side):
    """TriangleMesh's text formats (objects.h:343-400): z negated, v*a+b, 1-based indices."""
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for typ, text in MESH_TEXTS.items():
            path = os.path.join(d, f"t{typ}.txt")
            with open(path, "w") as fp:
                fp.write(text)
            if side == "ref":
                r = ob.Ref()
                r.add_mesh_file(path, 2.5, (1, -2, 3), (1, 1, 1), 0, 0, typ)
                out[f"type{typ}"] = r.mesh_triangles(0)
            else:
                out[f"type{typ}"] = ob.load_mesh_text(path, typ, 2.5, (1, -2, 3))
    return [np.frombuffer(t.encode(), np.uint8) for t in MESH_TEXTS.values()], out


def _eye_trace(e, side, org, dr, hs, ws):
    for i, (h, w) in enumerate(zip(hs, ws)):
        if side == "ref":
            e.trace(org[i], dr[i], (0, 0, 0), (1, 1, 1), True, int(w), int(h))
        else:
            e.trace(org[i], dr[i], (0, 0, 0), (1, 1, 1), True, int(w), int(h), path=i)


def _grid(W, H, step):
    hs, ws = np.meshgrid(np.arange(0, H, step), np.arange(0, W, step), indexing="ij")
    return hs.ravel(), ws.ravel()


def _sampling(ob, side):
    """sampling.h:11-43 through the rand() stream: eye hitpoints on the walls, then photons with four diffuse bounces each."""
    s = preset("walls_only")
    if side == "ref":
        e = ob.Ref(s)
        e.htable_new(1000001)
    else:
        e = ob.Oracle(s, RenderConfig(width=REF_W, height=REF_H, update_mode=0, into_rule=0))
    org, dr = camera_rays(REF_W, REF_H, 64)
    _eye_trace(e, side, org, dr, *_grid(REF_W, REF_H, 64))
    if side == "ref":
        e.seed(5)
    else:
        e.set_libc_rng(1, 5)
    rng = np.random.default_rng(1)
    pos, dirs = [], []
    for _ in range(4000):
        po = (rng.uniform(-2, 2), 19.999, 20 + rng.uniform(-2, 2))
        d = rng.normal(size=3)
        d /= np.linalg.norm(d)
        e.trace(po, d, (8796.0,) * 3, (1, 1, 1), False)
        pos.append(po)
        dirs.append(d)
    hp = e.download_hitpoints()
    assert hp["n"].sum() > 50
    return [np.array(pos), np.array(dirs)], {k: hp[k] for k in HP_FIELDS}


def _eye_pass(ob, side):
    """The oracle's eye_pass() (render() first half, main.cpp:185-219) == the reference's trace() per pixel, rows 300..329."""
    s = preset("c2_bunny_chess")
    if side == "ref":
        r = ob.Ref(s)
        assert r.image_size() == (REF_W, REF_H)
        r.htable_new(1000001)
        org, dr = camera_rays(REF_W, REF_H, 1)
        for h in range(300, 330):
            for w in range(REF_W):
                i = h * REF_W + w
                r.trace(org[i], dr[i], (0, 0, 0), (1, 1, 1), True, w, h)
        hp = r.download_hitpoints()
    else:
        o = ob.Oracle(s, RenderConfig(width=REF_W, height=REF_H, into_rule=0, consume_dof_rng=0))
        o.eye_pass(300, 330)
        hp = o.download_hitpoints()
    assert len(hp["pos"]) > 30 * REF_W
    return [], {k: hp[k] for k in ("key", "hw", "pos", "normal", "f", "r2")}


def _mirror(ob, side):
    """The mirror branch of trace() (main.cpp:129-134) on c1_mirror: eye rays on every 8th pixel, then 6000 photons aimed at the mirror."""
    s = preset("c1_mirror")
    if side == "ref":
        e = ob.Ref(s)
        assert e.image_size() == (REF_W, REF_H)
        e.htable_new(1000001)
    else:
        e = ob.Oracle(s, RenderConfig(width=REF_W, height=REF_H, update_mode=0, into_rule=0))
    org, dr = camera_rays(REF_W, REF_H, 8)
    _eye_trace(e, side, org, dr, *_grid(REF_W, REF_H, 8))
    if side == "ref":
        e.seed(31)
    else:
        e.set_libc_rng(1, 31)
    rng = np.random.default_rng(8)
    n = 6000
    po = np.stack([rng.uniform(-2, 2, n), np.full(n, 19.999), 20 + rng.uniform(-2, 2, n)], -1)
    tgt = np.array([-8.0, -13.0, 25.0]) + rng.uniform(-5, 5, (n, 3))
    pd = tgt - po
    pd /= np.linalg.norm(pd, axis=1)[:, None]
    f0 = 700.0 * (3.14159265358979 * 4.0)
    for i in range(n):
        e.trace(po[i], pd[i], (f0,) * 3, (1, 1, 1), False)
    hp = e.download_hitpoints()
    assert hp["n"].sum() > 1000
    return [po, pd], {k: hp[k] for k in HP_FIELDS}


CASES = {"bezier": _bezier, "mesh_loader": _mesh_loader, "sampling": _sampling, "eye_pass": _eye_pass, "mirror": _mirror}


def sample_rows(n):
    return np.arange(n) if n <= SAMPLE_ROWS else np.sort(np.random.default_rng(0).choice(n, SAMPLE_ROWS, replace=False))


def fixture_entries(name, inputs, outputs):
    """The arrays make_golden_live.py stores for one case."""
    g = {f"{name}__inputs_sha256": np.array(digest(inputs))}
    for k, a in outputs.items():
        rows = sample_rows(len(a))
        g[f"{name}__{k}__sha256"] = np.array(digest([a]))
        g[f"{name}__{k}__shape"] = np.array(a.shape, np.int64)
        g[f"{name}__{k}__rows"] = rows
        g[f"{name}__{k}__sample"] = a[rows]
    return g


@pytest.fixture(scope="module")
def G():
    return np.load(GOLDEN)


def _assert_matches(G, name, inputs, outputs):
    assert digest(inputs) == str(G[f"{name}__inputs_sha256"]), "the inputs differ from the stored ones (numpy's random stream?)"
    keys = sorted(k.split("__")[1] for k in G.files if k.startswith(f"{name}__") and k.endswith("__sha256") and "inputs" not in k)
    assert keys == sorted(outputs)
    for k, a in outputs.items():
        assert tuple(a.shape) == tuple(G[f"{name}__{k}__shape"]), k
        assert np.array_equal(a[G[f"{name}__{k}__rows"]], G[f"{name}__{k}__sample"]), k
        assert digest([a]) == str(G[f"{name}__{k}__sha256"]), k


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_equals_the_stored_reference_outputs(oracle_lib, G, name):
    _assert_matches(G, name, *CASES[name](oracle_lib, "oracle"))


@pytest.mark.ref
@pytest.mark.parametrize("name", sorted(CASES))
def test_stored_outputs_equal_the_live_reference(oracle_lib, G, name):
    _assert_matches(G, name, *CASES[name](oracle_lib, "ref"))
