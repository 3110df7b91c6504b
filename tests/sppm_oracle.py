"""ctypes wrapper of tests/sppm_oracle.cpp, the CPU reference of stochastic progressive photon mapping (SPPM). TEST INFRASTRUCTURE ONLY.

The library is compiled once per process into a temporary directory (the tree may be read-only), with the flags of oracle/Makefile:
no FMA contraction, so that its fp64 arithmetic is the GPU's bit for bit. Method names mirror cgraytracing_b200.Context."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sppm_oracle.cpp")
CXXFLAGS = ["-O2", "-fopenmp", "-ffp-contract=off", "-fPIC", "-shared", "-Wall", "-Wno-misleading-indentation"]

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_up = C.POINTER(C.c_uint32)
c_u8p = C.POINTER(C.c_uint8)

_lib = None


def lib():
    global _lib
    if _lib is None:
        out_dir = tempfile.mkdtemp(prefix="sppm_oracle_")
        so = os.path.join(out_dir, "libsppm_oracle.so")
        env = dict(os.environ)
        env.pop("CXX", None)
        env.pop("CC", None)
        subprocess.check_call([shutil.which("g++") or "g++"] + CXXFLAGS + ["-o", so, SRC], env=env)
        L = C.CDLL(so)
        L.sppm_create.restype = C.c_void_p
        L.sppm_destroy.argtypes = [C.c_void_p]
        L.sppm_num_visible.restype = C.c_int64
        L.sppm_num_visible.argtypes = [C.c_void_p]
        _lib = L
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


class SppmOracle:
    """One scene + SPPM state: mode 1 jitter, 2 corner (include/cgrt.h CGRT_SPPM_*). Per round: begin_round(r) -> photon_pass -> round_update."""

    def __init__(self, scene, cfg, mode):
        from oracle.binding import OrcConfig

        self.L = lib()
        k = OrcConfig()
        for f in ("width", "height", "max_depth", "num_of_samples", "use_dof", "consume_dof_rng", "hashsize", "update_mode", "into_rule"):
            setattr(k, f, int(getattr(cfg, f)))
        k.alpha, k.focus_plane, k.lens_radius = cfg.alpha, cfg.focus_plane, cfg.lens_radius
        k.lightorg = (C.c_double * 3)(*cfg.lightorg)
        k.camorg = (C.c_double * 3)(*cfg.camorg)
        k.seed = cfg.seed
        h = self.L.sppm_create(C.byref(k), int(mode))
        if not h:
            raise ValueError(f"SPPM mode must be 1 (jitter) or 2 (corner), got {mode}")
        self.h = C.c_void_p(h)
        self.cfg = cfg
        scene.build_into(self)

    def close(self):
        if self.h:
            self.L.sppm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- scene (SceneDesc.build_into)
    def add_texture(self, rgb, n, p, lenx, leny, isbump):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        return self.L.sppm_add_texture(self.h, _p(rgb, c_u8p), w, h, _p(_d(n), c_dp), _p(_d(p), c_dp), C.c_double(lenx), C.c_double(leny), int(isbump))

    def add_sphere(self, c, r, col, refl, transp):
        return self.L.sppm_add_sphere(self.h, _p(_d(c), c_dp), C.c_double(r), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    def add_plane(self, p, n, col, refl, transp, tex):
        return self.L.sppm_add_plane(self.h, _p(_d(p), c_dp), _p(_d(n), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(tex))

    def add_mesh(self, tri9, col, refl, transp, objtype):
        t = _d(tri9).reshape(-1, 9)
        return self.L.sppm_add_mesh(self.h, _p(t, c_dp), len(t), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(objtype))

    def add_bezier(self, cp, pos, col, refl, transp):
        cp = _d(cp).reshape(-1, 3)
        return self.L.sppm_add_bezier(self.h, _p(cp, c_dp), len(cp), _p(_d(pos), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp))

    # -- rounds
    def begin_round(self, r, nthreads=1):
        self.L.sppm_begin_round(self.h, C.c_uint32(r), int(nthreads))

    def photon_pass(self, first, count, nthreads=1):
        assert self.L.sppm_photon_pass(self.h, C.c_uint64(first), C.c_uint64(count), int(nthreads)) == 0

    def round_update(self):
        assert self.L.sppm_fold(self.h) == 0

    def download_hitpoints(self):
        """The round's visible points in canonical order: pos, r2, hw (pixel h, w), key (bucket), dflux / m (the round's accumulators)."""
        n = int(self.L.sppm_num_visible(self.h))
        o = dict(pos=np.zeros((n, 3)), r2=np.zeros(n), hw=np.zeros((n, 2), np.int32), key=np.zeros(n, np.uint32), dflux=np.zeros((n, 3)),
                 m=np.zeros(n, np.int32))
        self.L.sppm_download_visible(self.h, _p(o["pos"], c_dp), _p(o["r2"], c_dp), _p(o["hw"], c_ip), _p(o["key"], c_up), _p(o["dflux"], c_dp),
                                     _p(o["m"], c_ip))
        return o

    def download_pixels(self):
        H, W = self.cfg.height, self.cfg.width
        o = dict(tau=np.zeros((H, W, 3)), r2=np.zeros((H, W)), n=np.zeros((H, W), np.int32))
        self.L.sppm_download_pixels(self.h, _p(o["tau"], c_dp), _p(o["r2"], c_dp), _p(o["n"], c_ip))
        return o

    def gather_image(self, n_emitted):
        img = np.zeros((self.cfg.height, self.cfg.width, 3))
        self.L.sppm_gather_image(self.h, C.c_double(n_emitted), _p(img, c_dp))
        return img
