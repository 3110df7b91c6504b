"""ctypes bindings for the CPU oracle (oracle/liborc.so) and, when present, the compiled reference
(oracle/_ref/libcgref.so). TEST INFRASTRUCTURE ONLY — imported by tests/, __graft_entry__.smoke() and the
CPU-baseline legs of bench.py; never by the product package."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORC_SO = os.path.join(HERE, "liborc.so")
REF_SO = os.path.join(HERE, "_ref", "libcgref.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_up = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)
c_u8p = C.POINTER(C.c_uint8)


def build(force: bool = False) -> None:
    """make -C oracle (oracle always; _ref only where /root/reference exists)."""
    if force or not os.path.exists(ORC_SO) or os.path.getmtime(ORC_SO) < max(
        os.path.getmtime(os.path.join(HERE, f)) for f in ("oracle_capi.cpp", "ppm_oracle.hpp")
    ):
        subprocess.check_call(["make", "-C", HERE, "-s"])


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


class OrcConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("max_depth", C.c_int32), ("num_of_samples", C.c_int32),
        ("use_dof", C.c_int32), ("consume_dof_rng", C.c_int32), ("hashsize", C.c_int32), ("update_mode", C.c_int32),
        ("into_rule", C.c_int32), ("pad", C.c_int32),
        ("alpha", C.c_double), ("focus_plane", C.c_double), ("lens_radius", C.c_double),
        ("lightorg", C.c_double * 3), ("camorg", C.c_double * 3), ("seed", C.c_uint64),
    ]


class OrcCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "eye_segments", "photon_segments", "diffuse_hits", "bucket_probes", "nonempty_probes", "candidates", "deposits",
        "misses", "node_visits", "tri_tests")]


_orc = None


def orc_lib():
    global _orc
    if _orc is None:
        build()
        L = C.CDLL(ORC_SO)
        L.orc_create.restype = C.c_void_p
        L.orc_destroy.argtypes = [C.c_void_p]
        L.orc_num_hitpoints.restype = C.c_int64
        L.orc_num_hitpoints.argtypes = [C.c_void_p]
        L.orc_texture_height.restype = C.c_double
        L.orc_texture_height.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.orc_hash.restype = C.c_uint32
        _orc = L
    return _orc


class Oracle:
    """One oracle scene + renderer state. Method names mirror cgraytracing_b200.Context."""

    def __init__(self, scene=None, config=None):
        self.L = orc_lib()
        self.h = C.c_void_p(self.L.orc_create())
        self.cfg = None
        if config is not None:
            self.set_config(config)
        if scene is not None:
            scene.build_into(self)

    def close(self):
        if self.h:
            self.L.orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration
    def set_config(self, cfg):
        k = OrcConfig()
        for f in ("width", "height", "max_depth", "num_of_samples", "use_dof", "consume_dof_rng", "hashsize", "update_mode", "into_rule"):
            setattr(k, f, int(getattr(cfg, f)))
        k.alpha, k.focus_plane, k.lens_radius = cfg.alpha, cfg.focus_plane, cfg.lens_radius
        k.lightorg = (C.c_double * 3)(*cfg.lightorg)
        k.camorg = (C.c_double * 3)(*cfg.camorg)
        k.seed = cfg.seed
        self.cfg = cfg
        self.L.orc_set_config(self.h, C.byref(k))

    def set_libc_rng(self, on, seed=1):
        self.L.orc_set_libc_rng(self.h, C.c_int(int(on)), C.c_uint64(seed))

    # -- scene
    def add_texture(self, rgb, n, p, lenx, leny, isbump):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        return self.L.orc_add_texture(self.h, _p(rgb, c_u8p), w, h, _p(_d(n), c_dp), _p(_d(p), c_dp), C.c_double(lenx), C.c_double(leny), int(isbump))

    def add_sphere(self, c, r, col, refl, transp):
        return self.L.orc_add_sphere(self.h, _p(_d(c), c_dp), C.c_double(r), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    def add_plane(self, p, n, col, refl, transp, tex):
        return self.L.orc_add_plane(self.h, _p(_d(p), c_dp), _p(_d(n), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(tex))

    def add_mesh(self, tri9, col, refl, transp, objtype):
        t = _d(tri9).reshape(-1, 9)
        return self.L.orc_add_mesh(self.h, _p(t, c_dp), len(t), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(objtype))

    def add_bezier(self, cp, pos, col, refl, transp):
        cp = _d(cp).reshape(-1, 3)
        return self.L.orc_add_bezier(self.h, _p(cp, c_dp), len(cp), _p(_d(pos), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    def bump_triangles(self, obj):
        n = self.L.orc_bump_triangles(self.h, obj, None, 0)
        out = np.zeros((max(n, 0), 9))
        if n > 0:
            self.L.orc_bump_triangles(self.h, obj, _p(out, c_dp), n)
        return out

    # -- unit hooks
    def intersect_batch(self, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        t = np.zeros(n); nrm = np.zeros((n, 3)); raw = np.zeros((n, 3))
        obj = np.zeros(n, np.int32); into = np.zeros(n, np.int32); prim = np.zeros(n, np.int32)
        self.L.orc_intersect_batch(self.h, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(t, c_dp), _p(nrm, c_dp), _p(raw, c_dp),
                                   _p(obj, c_ip), _p(into, c_ip), _p(prim, c_ip))
        return dict(t=t, nrm=nrm, nrm_raw=raw, obj=obj, into=into, prim=prim)

    def object_intersect(self, objid, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        hit = np.zeros(n, np.int32); ln = np.zeros(n); nrm = np.zeros((n, 3))
        self.L.orc_object_intersect(self.h, objid, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(hit, c_ip), _p(ln, c_dp), _p(nrm, c_dp))
        return hit, ln, nrm

    def mesh_brute(self, objid, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        hit = np.zeros(n, np.int32); ln = np.zeros(n); tri = np.zeros(n, np.int32)
        r = self.L.orc_mesh_brute(self.h, objid, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(hit, c_ip), _p(ln, c_dp), _p(tri, c_ip))
        assert r == 0
        return hit, ln, tri

    def surface_color(self, objid, pos):
        pos = _d(pos).reshape(-1, 3)
        col = np.zeros_like(pos)
        self.L.orc_surface_color(self.h, objid, C.c_int64(len(pos)), _p(pos, c_dp), _p(col, c_dp))
        return col

    def texture_color(self, tex, pos):
        pos = _d(pos).reshape(-1, 3)
        n = len(pos)
        hit = np.zeros(n, np.int32); col = np.zeros((n, 3)); rc = np.zeros((n, 2), np.int32)
        self.L.orc_texture_color(self.h, tex, C.c_int64(n), _p(pos, c_dp), _p(hit, c_ip), _p(col, c_dp), _p(rc, c_ip))
        return hit, col, rc

    def texture_height(self, tex, i, j):
        return self.L.orc_texture_height(self.h, tex, i, j)

    def bezier_eval(self, objid, what, paras, org=(0, 0, 0), dir=(0, 0, 0)):
        out = np.zeros(3)
        r = self.L.orc_bezier_eval(self.h, objid, what, _p(_d(paras), c_dp), _p(_d(org), c_dp), _p(_d(dir), c_dp), _p(out, c_dp))
        assert r == 0
        return out

    # -- passes
    def trace(self, org, dir, flux, adj, flag, x=0, y=0, path=0):
        self.L.orc_trace(self.h, _p(_d(org), c_dp), _p(_d(dir), c_dp), _p(_d(flux), c_dp), _p(_d(adj), c_dp), int(flag), x, y, C.c_uint64(path))

    def eye_pass(self, y0=0, y1=-1, nthreads=1):
        """nthreads > 1 (Philox mode): rows traced in parallel, merged in the reference's creation order — same table."""
        if nthreads > 1:
            self.L.orc_eye_pass_mt(self.h, y0, y1, int(nthreads))
        else:
            self.L.orc_eye_pass(self.h, y0, y1)

    # -- stochastic PPM (Context.set_sppm): per round sppm_begin_round(r), or sppm_eye_pass -> export/import_hitpoints -> build_grid;
    #    then photon_pass -> round_update (the per-pixel fold) as in PPM
    def set_sppm(self, mode):
        """mode 0 off, 1 jitter, 2 corner (include/cgrt.h CGRT_SPPM_*), after set_config; resets the pixel statistics."""
        r = self.L.orc_set_sppm(self.h, int(mode))
        if r == -1:
            raise ValueError(f"SPPM mode must be 0 (off), 1 (jitter) or 2 (corner), got {mode}")
        if r:
            raise ValueError("SPPM needs the per-round update (update_mode=1)")

    def sppm_begin_round(self, r, nthreads=1):
        """A new table and round r's eye pass, every visible point at its pixel's radius."""
        assert self.L.orc_sppm_begin_round(self.h, C.c_uint32(r), int(nthreads)) == 0

    def sppm_eye_pass(self, r, y0=0, y1=-1, nthreads=1):
        """Round r's eye pass over rows [y0, y1) into the pending visible points; build_grid inserts them."""
        assert self.L.orc_sppm_eye_pass(self.h, C.c_uint32(r), int(y0), int(y1), int(nthreads)) == 0

    def build_grid(self):
        """SPPM: the pending visible points into the round's table in canonical order. PPM: nothing to do."""
        assert self.L.orc_build_grid(self.h) == 0

    def sppm_download_pixels(self):
        H, W = self.cfg.height, self.cfg.width
        o = dict(tau=np.zeros((H, W, 3)), r2=np.zeros((H, W)), n=np.zeros((H, W), np.int32))
        self.L.orc_sppm_download_pixels(self.h, _p(o["tau"], c_dp), _p(o["r2"], c_dp), _p(o["n"], c_ip))
        return o

    def num_hitpoints(self):
        return int(self.L.orc_num_hitpoints(self.h))

    def download_hitpoints(self, fields=None):
        n = self.num_hitpoints()
        spec = dict(pos=((n, 3), np.float64), normal=((n, 3), np.float64), f=((n, 3), np.float64), flux=((n, 3), np.float64), r2=((n,), np.float64),
                    n=((n,), np.int32), hw=((n, 2), np.int32), key=((n,), np.uint32), seq=((n,), np.uint32), code=((n,), np.uint32),
                    path=((n,), np.uint64))
        o = {k: np.zeros(sh, dt) for k, (sh, dt) in spec.items() if fields is None or k in fields}
        g = o.get
        self.L.orc_download_hitpoints(self.h, _p(g("pos"), c_dp), _p(g("normal"), c_dp), _p(g("f"), c_dp), _p(g("flux"), c_dp),
                                      _p(g("r2"), c_dp), _p(g("n"), c_ip), _p(g("hw"), c_ip), _p(g("key"), c_up), _p(g("seq"), c_up),
                                      _p(g("code"), c_up), _p(g("path"), c_u64p))
        return o

    def download_accum(self):
        n = self.num_hitpoints()
        df = np.zeros((n, 3)); m = np.zeros(n, np.int32)
        self.L.orc_download_accum(self.h, _p(df, c_dp), _p(m, c_ip))
        return df, m

    def upload_accum(self, dflux, m):
        df = _d(dflux).reshape(-1, 3); mm = np.ascontiguousarray(m, dtype=np.int32)
        assert len(df) == len(mm) == self.num_hitpoints()
        self.L.orc_upload_accum(self.h, _p(df, c_dp), _p(mm, c_ip))

    def export_hitpoints(self):
        """-> float64 [n, 12] records in the GPU path's exchange format (cgrt_export_hitpoints_dev); under SPPM, between sppm_eye_pass and
        build_grid, of the pending visible points."""
        self.L.orc_export_hitpoints.restype = C.c_int64
        n = self.L.orc_export_hitpoints(self.h, None)
        rec = np.zeros((n, 12))
        if n:
            self.L.orc_export_hitpoints(self.h, _p(rec, c_dp))
        return rec

    def import_hitpoints(self, rec):
        rec = _d(rec).reshape(-1, 12)
        assert self.L.orc_import_hitpoints(self.h, C.c_int64(len(rec)), _p(rec, c_dp)) == 0

    def photon_pass(self, first, count, nthreads=1):
        sec = C.c_double(0)
        r = self.L.orc_photon_pass(self.h, C.c_uint64(first), C.c_uint64(count), int(nthreads), C.byref(sec))
        assert r == 0, r
        return sec.value

    def round_update(self):
        assert self.L.orc_round_update(self.h) == 0

    def gather_image(self, n_emitted):
        img = np.zeros((self.cfg.height, self.cfg.width, 3))
        self.L.orc_gather_image(self.h, C.c_double(n_emitted), _p(img, c_dp))
        return img

    def counters(self):
        k = OrcCounters()
        self.L.orc_get_counters(self.h, C.byref(k))
        return {n: int(getattr(k, n)) for n, _ in OrcCounters._fields_}

    def max_threads(self):
        """Host threads the oracle may use: the CPUs this process may run on, NOT omp_get_max_threads() — launchers such as
        torch.distributed.run export OMP_NUM_THREADS=1 into every rank, which would silently time the CPU arm on one core."""
        try:
            return max(1, len(os.sched_getaffinity(0)))
        except AttributeError:
            return max(1, os.cpu_count() or 1)


def hash_keys(pos, hashsize, celllength_in):
    pos = _d(pos).reshape(-1, 3)
    n = len(pos)
    key = np.zeros(n, np.uint32); ixyz = np.zeros((n, 3), np.int32)
    orc_lib().orc_hash_keys(C.c_int64(n), _p(pos, c_dp), int(hashsize), C.c_double(celllength_in), _p(key, c_up), _p(ixyz, c_ip))
    return key, ixyz


def grid_params(hashsize, celllength_in):
    cells = C.c_int(0); cl = C.c_double(0)
    orc_lib().orc_grid_params(int(hashsize), C.c_double(celllength_in), C.byref(cells), C.byref(cl))
    return cells.value, cl.value


def hash3(ix, iy, iz, hashsize):
    return int(orc_lib().orc_hash(int(ix), int(iy), int(iz), int(hashsize)))


def philox(ctr, key):
    c = np.asarray(ctr, np.uint32); k = np.asarray(key, np.uint32); o = np.zeros(4, np.uint32)
    orc_lib().orc_philox(_p(c, c_up), _p(k, c_up), _p(o, c_up))
    return o


def sample(seed, pass_id, path, dim, what, aux=(0, 0, 0)):
    out = np.zeros(3)
    orc_lib().orc_sample(C.c_uint64(seed), C.c_uint32(pass_id), C.c_uint64(path), C.c_uint32(dim), int(what), _p(_d(aux), c_dp), _p(out, c_dp))
    return out


def gamma_corr(x):
    x = _d(x).ravel()
    out = np.zeros(len(x), np.int32)
    orc_lib().orc_gamma_corr(C.c_int64(len(x)), _p(x, c_dp), _p(out, c_ip))
    return out


def tonemap_flip(img):
    h, w = img.shape[:2]
    out = np.zeros((h, w, 3), np.uint8)
    orc_lib().orc_tonemap_flip(w, h, _p(_d(img), c_dp), _p(out, c_u8p))
    return out


def average_u8(images):
    """average.cpp: per byte, sum of img/n over the n images."""
    imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
    n = len(imgs)
    ptrs = (c_u8p * n)(*[_p(im, c_u8p) for im in imgs])
    out = np.zeros(imgs[0].shape, np.uint8)
    orc_lib().orc_average_u8(n, ptrs, C.c_int64(imgs[0].size), _p(out, c_u8p))
    return out


def det_inv(a, b, c):
    d = C.c_double(0); inv9 = np.zeros(9)
    ok = orc_lib().orc_det_inv(_p(_d(a), c_dp), _p(_d(b), c_dp), _p(_d(c), c_dp), C.byref(d), _p(inv9, c_dp))
    return d.value, bool(ok), inv9.reshape(3, 3)


def load_mesh_text(filename, typeofdata, a, b):
    L = orc_lib()
    n = L.orc_load_mesh_text(filename.encode(), int(typeofdata), C.c_double(a), _p(_d(b), c_dp), None, 0)
    if n < 0:
        raise FileNotFoundError(filename)
    out = np.zeros((n, 9))
    L.orc_load_mesh_text(filename.encode(), int(typeofdata), C.c_double(a), _p(_d(b), c_dp), _p(out, c_dp), n)
    return out


# ---------------------------------------------------------------------------------------------------------------
# The compiled reference (only where oracle/_ref/libcgref.so exists)
# ---------------------------------------------------------------------------------------------------------------
def have_ref() -> bool:
    return os.path.exists(REF_SO)


def write_type0_mesh(path, tri9):
    """Write world-space triangles in the reference's type-0 text format so that TriangleMesh(file, a=1, b=0, type 0)
    reloads them bit-exactly: the loader negates z (objects.h:348), so z is pre-negated; %.17g round-trips fp64."""
    t = np.asarray(tri9, dtype=np.float64).reshape(-1, 3, 3)
    with open(path, "w") as fp:
        for tri in t:
            fp.write("begin\n")
            for v in tri:
                fp.write("vertex %.17g %.17g %.17g\n" % (v[0], v[1], -v[2]))
            fp.write("end\n\n")


class Ref:
    """The reference's own classes and trace() (global scene inside libcgref.so — one instance at a time)."""

    def __init__(self, scene=None):
        L = C.CDLL(REF_SO)
        L.ref_hash.restype = C.c_uint32
        L.ref_texture_height.restype = C.c_double
        L.ref_num_hitpoints.restype = C.c_int64
        L.ref_stbi_load.restype = c_u8p
        self.L = L
        self.tmp = tempfile.mkdtemp(prefix="cgref_")
        L.ref_reset()
        if scene is not None:
            scene.build_into(self)

    def seed(self, s):
        self.L.ref_seed(C.c_uint64(s))

    def add_texture(self, rgb, n, p, lenx, leny, isbump):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        return self.L.ref_add_texture(_p(rgb, c_u8p), w, h, _p(_d(n), c_dp), _p(_d(p), c_dp), C.c_double(lenx), C.c_double(leny), int(isbump))

    def add_sphere(self, c, r, col, refl, transp):
        return self.L.ref_add_sphere(_p(_d(c), c_dp), C.c_double(r), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    def add_plane(self, p, n, col, refl, transp, tex):
        return self.L.ref_add_plane(_p(_d(p), c_dp), _p(_d(n), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(tex))

    def add_mesh(self, tri9, col, refl, transp, objtype):
        # TriangleMesh only reads files: round-trip through a type-0 file; objtype 2 keeps its flag via a type-2 file
        t = np.asarray(tri9, dtype=np.float64).reshape(-1, 9)
        path = os.path.join(self.tmp, "mesh%d.txt" % len(os.listdir(self.tmp)))
        if objtype == 2:
            v = t.reshape(-1, 3)
            with open(path, "w") as fp:
                fp.write("%d\n" % len(v))
                for q in v:
                    fp.write("v %.17g %.17g %.17g\n" % (q[0], q[1], -q[2]))
                fp.write("%d\n" % len(t))
                for i in range(len(t)):
                    a = 3 * i + 1
                    fp.write("f %d/%d/%d %d/%d/%d %d/%d/%d \n" % (a, a, a, a + 1, a + 1, a + 1, a + 2, a + 2, a + 2))
            return self.add_mesh_file(path, 1.0, (0, 0, 0), col, refl, transp, 2)
        write_type0_mesh(path, t)
        return self.add_mesh_file(path, 1.0, (0, 0, 0), col, refl, transp, 0)

    def add_mesh_file(self, filename, a, b, col, refl, transp, typeofdata):
        import sys
        sys.stdout.flush()
        # the reference loader freopen()s stdin and fclose()s it (objects.h:342,401); keep fd 0 alive across the call
        saved = os.dup(0)
        try:
            r = self.L.ref_add_mesh_file(filename.encode(), C.c_double(a), _p(_d(b), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(typeofdata))
        finally:
            os.dup2(saved, 0)
            os.close(saved)
        return r

    def add_bezier(self, cp, pos, col, refl, transp):
        cp = _d(cp).reshape(-1, 3)
        return self.L.ref_add_bezier(_p(cp, c_dp), len(cp), _p(_d(pos), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    def mesh_triangles(self, objid):
        n = self.L.ref_mesh_triangles(objid, None, 0)
        out = np.zeros((max(n, 0), 9))
        if n > 0:
            self.L.ref_mesh_triangles(objid, _p(out, c_dp), n)
        return out

    def hash3(self, ix, iy, iz, hashsize):
        return int(self.L.ref_hash(int(ix), int(iy), int(iz), int(hashsize)))

    def hash_keys(self, pos, hashsize, celllength_in):
        pos = _d(pos).reshape(-1, 3)
        n = len(pos)
        key = np.zeros(n, np.uint32); ixyz = np.zeros((n, 3), np.int32)
        cells = C.c_int(0); cl = C.c_double(0)
        self.L.ref_hash_keys(C.c_int64(n), _p(pos, c_dp), int(hashsize), C.c_double(celllength_in), _p(key, c_up), _p(ixyz, c_ip), C.byref(cells), C.byref(cl))
        return key, ixyz, cells.value, cl.value

    def object_intersect(self, objid, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        hit = np.zeros(n, np.int32); ln = np.zeros(n); nrm = np.zeros((n, 3))
        self.L.ref_object_intersect(objid, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(hit, c_ip), _p(ln, c_dp), _p(nrm, c_dp))
        return hit, ln, nrm

    def triangle_intersect(self, tri9, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        hit = np.zeros(n, np.int32); ln = np.zeros(n); nrm = np.zeros((n, 3))
        self.L.ref_triangle_intersect(_p(_d(tri9).ravel(), c_dp), C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(hit, c_ip), _p(ln, c_dp), _p(nrm, c_dp))
        return hit, ln, nrm

    def intersect_batch(self, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        t = np.zeros(n); nrm = np.zeros((n, 3)); raw = np.zeros((n, 3)); obj = np.zeros(n, np.int32); into = np.zeros(n, np.int32)
        self.L.ref_intersect_batch(C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(t, c_dp), _p(nrm, c_dp), _p(raw, c_dp), _p(obj, c_ip), _p(into, c_ip))
        return dict(t=t, nrm=nrm, nrm_raw=raw, obj=obj, into=into)

    def surface_color(self, objid, pos):
        pos = _d(pos).reshape(-1, 3)
        col = np.zeros_like(pos)
        self.L.ref_surface_color(objid, C.c_int64(len(pos)), _p(pos, c_dp), _p(col, c_dp))
        return col

    def texture_color(self, tex, pos):
        pos = _d(pos).reshape(-1, 3)
        n = len(pos)
        hit = np.zeros(n, np.int32); col = np.zeros((n, 3))
        self.L.ref_texture_color(tex, C.c_int64(n), _p(pos, c_dp), _p(hit, c_ip), _p(col, c_dp))
        return hit, col

    def texture_height(self, tex, i, j):
        return self.L.ref_texture_height(tex, i, j)

    def bezier_eval(self, objid, what, paras, org=(0, 0, 0), dir=(0, 0, 0)):
        out = np.zeros(3)
        r = self.L.ref_bezier_eval(objid, what, _p(_d(paras), c_dp), _p(_d(org), c_dp), _p(_d(dir), c_dp), _p(out, c_dp))
        assert r == 0
        return out

    def gamma_corr(self, x):
        x = _d(x).ravel()
        out = np.zeros(len(x), np.int32)
        self.L.ref_gamma_corr(C.c_int64(len(x)), _p(x, c_dp), _p(out, c_ip))
        return out

    def det_inv(self, a, b, c):
        d = C.c_double(0); inv9 = np.zeros(9)
        ok = self.L.ref_det_inv(_p(_d(a), c_dp), _p(_d(b), c_dp), _p(_d(c), c_dp), C.byref(d), _p(inv9, c_dp))
        return d.value, bool(ok), inv9.reshape(3, 3)

    def sample(self, what, aux=(0, 0, 0)):
        out = np.zeros(3)
        self.L.ref_sample(int(what), _p(_d(aux), c_dp), _p(out, c_dp))
        return out

    def htable_new(self, hashsize=1000001):
        self.L.ref_htable_new(int(hashsize))

    def trace(self, org, dir, flux, adj, flag, x=0, y=0):
        self.L.ref_trace(_p(_d(org), c_dp), _p(_d(dir), c_dp), _p(_d(flux), c_dp), _p(_d(adj), c_dp), int(flag), x, y)

    def num_hitpoints(self):
        return int(self.L.ref_num_hitpoints())

    def download_hitpoints(self):
        n = self.num_hitpoints()
        o = dict(pos=np.zeros((n, 3)), normal=np.zeros((n, 3)), f=np.zeros((n, 3)), flux=np.zeros((n, 3)), r2=np.zeros(n),
                 n=np.zeros(n, np.int32), hw=np.zeros((n, 2), np.int32), key=np.zeros(n, np.uint32))
        self.L.ref_download_hitpoints(_p(o["pos"], c_dp), _p(o["normal"], c_dp), _p(o["f"], c_dp), _p(o["flux"], c_dp), _p(o["r2"], c_dp),
                                      _p(o["n"], c_ip), _p(o["hw"], c_ip), _p(o["key"], c_up))
        return o

    def image_size(self):
        return self.L.ref_image_width(), self.L.ref_image_height()

    def eye_pass_as_shipped(self):
        """main.cpp:185-219 over the compiled-in image through the reference's own trace()."""
        self.L.ref_eye_pass_as_shipped()

    def photon_loop_as_shipped(self, num_photon, num_threads=8, seed=1):
        """main.cpp:222-249: every one of `num_threads` threads traces `num_photon` photons (glibc rand() and its lock). -> seconds"""
        self.L.ref_photon_loop_as_shipped.restype = C.c_double
        return float(self.L.ref_photon_loop_as_shipped(int(num_photon), int(num_threads), C.c_uint(seed)))
