"""ctypes binding of the C ABI (include/cgrt.h -> cgraytracing_b200/libcgrt.so).

This is host plumbing only: every number on the hot path is computed by the CUDA kernels behind the ABI. There is no
CPU fallback: if the shared library is missing or no GPU is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libcgrt.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int32)
c_up = C.POINTER(C.c_uint32)
c_u64p = C.POINTER(C.c_uint64)
c_u8p = C.POINTER(C.c_uint8)

# every symbol include/cgrt.h declares (tests/test_abi.py checks the header against this list and the library)
ABI_SYMBOLS = [
    "cgrt_create", "cgrt_destroy", "cgrt_last_error", "cgrt_version", "cgrt_default_config", "cgrt_set_config", "cgrt_get_stream",
    "cgrt_synchronize", "cgrt_add_texture", "cgrt_add_sphere", "cgrt_add_plane", "cgrt_add_mesh", "cgrt_add_bezier", "cgrt_commit_scene",
    "cgrt_intersect_batch", "cgrt_hash_keys", "cgrt_surface_color", "cgrt_object_triangles", "cgrt_sample", "cgrt_radix_sort",
    "cgrt_count_traversal", "cgrt_eye_pass", "cgrt_export_hitpoints_dev", "cgrt_import_hitpoints_dev", "cgrt_build_grid", "cgrt_photon_pass",
    "cgrt_accum_dev", "cgrt_allreduce_accum", "cgrt_round_update", "cgrt_gather_image", "cgrt_num_hitpoints", "cgrt_download_hitpoints",
    "cgrt_download_accum", "cgrt_download_grid", "cgrt_get_counters", "cgrt_get_timings", "cgrt_set_counting", "cgrt_set_profiling", "cgrt_set_culling", "cgrt_set_overlap", "cgrt_average_u8", "cgrt_average_f64",
    "cgrt_check_guards", "cgrt_release_cached_memory", "cgrt_photon_chunk", "cgrt_deposit_record_bytes", "cgrt_trace",
    "cgrt_peer_export", "cgrt_peer_attach", "cgrt_comm_unique_id", "cgrt_comm_init_rank", "cgrt_comm_init_all", "cgrt_comm_destroy", "cgrt_allgather_hitpoints", "cgrt_set_comm",
    "cgrt_set_sppm", "cgrt_sppm_begin_round", "cgrt_sppm_download_pixels", "cgrt_sppm_eye_pass",
]


class CgrtConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32), ("max_depth", C.c_int32), ("num_of_samples", C.c_int32), ("use_dof", C.c_int32),
        ("hashsize", C.c_int32), ("accum_mode", C.c_int32), ("update_mode", C.c_int32),
        ("alpha", C.c_double), ("focus_plane", C.c_double), ("lens_radius", C.c_double),
        ("lightorg", C.c_double * 3), ("camorg", C.c_double * 3), ("seed", C.c_uint64),
    ]


class CgrtCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "eye_segments", "photon_segments", "diffuse_hits", "candidates", "deposits", "node_visits", "tri_tests", "hitpoints", "gpu_launches", "gathered_hits", "exact_tests",
        "cell_groups", "staged_candidates")]


class CgrtError(RuntimeError):
    pass


_lib = None


def load_library():
    """dlopen libcgrt.so. Raises (never falls back) when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CgrtError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`; there is no CPU fallback")
        L = C.CDLL(os.environ.get("CGRT_LIB", LIB_PATH))  # CGRT_LIB: dev override for A/B builds of the same library
        L.cgrt_last_error.restype = C.c_char_p
        L.cgrt_last_error.argtypes = [C.c_void_p]
        L.cgrt_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        for name in ABI_SYMBOLS:
            getattr(L, name)  # AttributeError if the library does not export it
        _lib = L
    return _lib


def _d(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


class Context:
    """One GPU context = one scene + one hitpoint set (cgrt_ctx). Methods map 1:1 onto the C ABI."""

    def __init__(self, device: int = 0, scene=None, config=None):
        self.L = load_library()
        h = C.c_void_p()
        rc = self.L.cgrt_create(int(device), C.byref(h))
        if rc != 0:
            raise CgrtError(f"cgrt_create(device={device}) failed with status {rc} (no usable CUDA device? there is no CPU fallback)")
        self.h = h
        self.cfg = None
        if config is not None:
            self.set_config(config)
        if scene is not None:
            scene.build_into(self)
            self.commit()

    # -- plumbing
    def _ck(self, rc):
        if rc != 0:
            raise CgrtError(f"status {rc}: {self.L.cgrt_last_error(self.h).decode()}")

    def close(self):
        if getattr(self, "h", None):
            self.L.cgrt_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def set_config(self, cfg, accum_mode=None):
        k = CgrtConfig()
        self.L.cgrt_default_config(C.byref(k))
        for f in ("width", "height", "max_depth", "num_of_samples", "use_dof", "hashsize"):
            setattr(k, f, int(getattr(cfg, f)))
        k.accum_mode = int(getattr(cfg, "accum_mode", 0) if accum_mode is None else accum_mode)
        k.update_mode = int(getattr(cfg, "update_mode", 1))  # 0: the reference's per-photon update (U1), 1: per round (U2)
        if k.update_mode == 0:
            k.accum_mode = 0  # the library keeps fp64 sums in that mode whatever is asked for; keep this side's view of the buffer in step
        k.alpha, k.focus_plane, k.lens_radius = cfg.alpha, cfg.focus_plane, cfg.lens_radius
        k.lightorg = (C.c_double * 3)(*cfg.lightorg)
        k.camorg = (C.c_double * 3)(*cfg.camorg)
        k.seed = cfg.seed
        self._ck(self.L.cgrt_set_config(self.h, C.byref(k)))
        self.cfg = cfg
        self.accum_mode = k.accum_mode

    def stream(self) -> int:
        s = C.c_void_p()
        self._ck(self.L.cgrt_get_stream(self.h, C.byref(s)))
        return s.value or 0

    def synchronize(self):
        self._ck(self.L.cgrt_synchronize(self.h))

    # -- scene (same argument meaning as the reference constructors)
    def add_texture(self, rgb, n, p, lenx, leny, isbump):
        rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
        h, w = rgb.shape[:2]
        tid = C.c_int(-1)
        self._ck(self.L.cgrt_add_texture(self.h, _p(rgb, c_u8p), w, h, _p(_d(n), c_dp), _p(_d(p), c_dp), C.c_double(lenx), C.c_double(leny), int(isbump), C.byref(tid)))
        return tid.value

    def add_sphere(self, c, r, col, refl=0.0, transp=0.0):
        oid = C.c_int(-1)
        self._ck(self.L.cgrt_add_sphere(self.h, _p(_d(c), c_dp), C.c_double(r), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), C.byref(oid)))
        return oid.value

    def add_plane(self, p, n, col, refl=0.0, transp=0.0, tex=-1):
        oid = C.c_int(-1)
        self._ck(self.L.cgrt_add_plane(self.h, _p(_d(p), c_dp), _p(_d(n), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(tex), C.byref(oid)))
        return oid.value

    def add_mesh(self, tri9, col, refl=0.0, transp=0.0, objtype=0):
        t = _d(tri9).reshape(-1, 9)
        oid = C.c_int(-1)
        self._ck(self.L.cgrt_add_mesh(self.h, _p(t, c_dp), len(t), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), int(objtype), C.byref(oid)))
        return oid.value

    def add_bezier(self, cp, pos, col, refl=0.0, transp=0.0):
        cp = _d(cp).reshape(-1, 3)
        oid = C.c_int(-1)
        self._ck(self.L.cgrt_add_bezier(self.h, _p(cp, c_dp), len(cp), _p(_d(pos), c_dp), _p(_d(col), c_dp), C.c_double(refl), C.c_double(transp), C.byref(oid)))
        return oid.value

    def commit(self):
        self._ck(self.L.cgrt_commit_scene(self.h))

    # -- parity hooks
    def intersect_batch(self, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        n = len(org)
        t = np.zeros(n); nrm = np.zeros((n, 3)); raw = np.zeros((n, 3))
        obj = np.zeros(n, np.int32); into = np.zeros(n, np.int32); prim = np.zeros(n, np.int32)
        self._ck(self.L.cgrt_intersect_batch(self.h, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(t, c_dp), _p(nrm, c_dp), _p(raw, c_dp),
                                             _p(obj, c_ip), _p(into, c_ip), _p(prim, c_ip)))
        return dict(t=t, nrm=nrm, nrm_raw=raw, obj=obj, into=into, prim=prim)

    def count_traversal(self, org, dir):
        org, dir = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3)
        nv, tt = C.c_uint64(0), C.c_uint64(0)
        self._ck(self.L.cgrt_count_traversal(self.h, C.c_int64(len(org)), _p(org, c_dp), _p(dir, c_dp), C.byref(nv), C.byref(tt)))
        return nv.value, tt.value

    def hash_keys(self, pos, hashsize, celllength_in):
        pos = _d(pos).reshape(-1, 3)
        n = len(pos)
        key = np.zeros(n, np.uint32); ixyz = np.zeros((n, 3), np.int32)
        self._ck(self.L.cgrt_hash_keys(self.h, C.c_int64(n), _p(pos, c_dp), int(hashsize), C.c_double(celllength_in), _p(key, c_up), _p(ixyz, c_ip)))
        return key, ixyz

    def surface_color(self, obj, pos):
        pos = _d(pos).reshape(-1, 3)
        col = np.zeros_like(pos)
        self._ck(self.L.cgrt_surface_color(self.h, int(obj), C.c_int64(len(pos)), _p(pos, c_dp), _p(col, c_dp)))
        return col

    def object_triangles(self, obj):
        n = C.c_int64(0)
        self._ck(self.L.cgrt_object_triangles(self.h, int(obj), None, C.c_int64(0), C.byref(n)))
        out = np.zeros((n.value, 9))
        if n.value:
            self._ck(self.L.cgrt_object_triangles(self.h, int(obj), _p(out, c_dp), C.c_int64(n.value), C.byref(n)))
        return out

    def sample(self, seed, pass_id, path, dim, what, aux=(0, 0, 0)):
        out = np.zeros(3)
        self._ck(self.L.cgrt_sample(self.h, C.c_uint64(seed), C.c_uint32(pass_id), C.c_uint64(path), C.c_uint32(dim), int(what), _p(_d(aux), c_dp), _p(out, c_dp)))
        return out

    def radix_sort(self, keys, nbits=64):
        keys = np.ascontiguousarray(keys, dtype=np.uint64)
        out = np.zeros_like(keys); perm = np.zeros(len(keys), np.uint32)
        self._ck(self.L.cgrt_radix_sort(self.h, C.c_int64(len(keys)), _p(keys, c_u64p), int(nbits), _p(out, c_u64p), _p(perm, c_up)))
        return out, perm

    # -- passes
    def eye_pass(self, y0=0, y1=-1):
        self._ck(self.L.cgrt_eye_pass(self.h, int(y0), int(y1)))

    def export_hitpoints_dev(self):
        ptr = C.c_void_p(); n = C.c_int64(0)
        self._ck(self.L.cgrt_export_hitpoints_dev(self.h, C.byref(ptr), C.byref(n)))
        return ptr.value or 0, n.value

    def import_hitpoints_dev(self, ptr, count):
        self._ck(self.L.cgrt_import_hitpoints_dev(self.h, C.c_void_p(ptr), C.c_int64(count)))

    def build_grid(self):
        self._ck(self.L.cgrt_build_grid(self.h))

    def photon_pass(self, first, count):
        self._ck(self.L.cgrt_photon_pass(self.h, C.c_uint64(first), C.c_uint64(count)))

    def trace(self, org, dir, weight, flag, depth=0, x=None, y=None, first_index=0):
        """trace() of main.cpp:42 for n rays: flag True = eye rays (weight = adj, pixels x, y; before build_grid), False = photons
        (weight = flux; after build_grid; ray k draws the random numbers of photon first_index + k)."""
        org, dir, weight = _d(org).reshape(-1, 3), _d(dir).reshape(-1, 3), _d(weight).reshape(-1, 3)
        n = len(org)
        xi = None if x is None else np.ascontiguousarray(x, dtype=np.int32)
        yi = None if y is None else np.ascontiguousarray(y, dtype=np.int32)
        self._ck(self.L.cgrt_trace(self.h, C.c_int64(n), _p(org, c_dp), _p(dir, c_dp), _p(weight, c_dp), int(bool(flag)), int(depth), _p(xi, c_ip), _p(yi, c_ip),
                                   C.c_uint64(first_index)))

    def accum_dev(self):
        ptr = C.c_void_p(); n = C.c_int64(0)
        self._ck(self.L.cgrt_accum_dev(self.h, C.byref(ptr), C.byref(n)))
        return ptr.value or 0, n.value

    def round_update(self):
        self._ck(self.L.cgrt_round_update(self.h))

    def gather_image(self, n_emitted, want_rgb8=False):
        img = np.zeros((self.cfg.height, self.cfg.width, 3))
        rgb8 = np.zeros((self.cfg.height, self.cfg.width, 3), np.uint8) if want_rgb8 else None
        self._ck(self.L.cgrt_gather_image(self.h, C.c_double(n_emitted), _p(img, c_dp), _p(rgb8, c_u8p)))
        return (img, rgb8) if want_rgb8 else img

    # -- stochastic progressive photon mapping
    def set_sppm(self, mode):
        """0 off (PPM), 1 jitter, 2 corner (include/cgrt.h CGRT_SPPM_*). After commit, before any eye pass."""
        self._ck(self.L.cgrt_set_sppm(self.h, int(mode)))

    def sppm_begin_round(self, r):
        """Eye pass of round r with its own camera stream, grid at the pixels' current radii."""
        self._ck(self.L.cgrt_sppm_begin_round(self.h, C.c_uint32(r)))

    def sppm_eye_pass(self, r, y0=0, y1=-1):
        """Eye pass of round r over rows [y0, y1) (y1 < 0: all rows) without the grid: exchange the records with the other ranks, then
        build_grid. sppm_eye_pass(r, 0, H) + build_grid() is sppm_begin_round(r)."""
        self._ck(self.L.cgrt_sppm_eye_pass(self.h, C.c_uint32(r), int(y0), int(y1)))

    def sppm_download_pixels(self):
        """-> dict tau [H, W, 3], r2 [H, W], n [H, W] (row h = image[h])."""
        H, W = self.cfg.height, self.cfg.width
        o = dict(tau=np.zeros((H, W, 3)), r2=np.zeros((H, W)), n=np.zeros((H, W), np.int32))
        self._ck(self.L.cgrt_sppm_download_pixels(self.h, _p(o["tau"], c_dp), _p(o["r2"], c_dp), _p(o["n"], c_ip)))
        return o

    # -- multi-run averaging (average.cpp)
    def average_u8(self, images):
        imgs = [np.ascontiguousarray(im, dtype=np.uint8) for im in images]
        n, nbytes = len(imgs), imgs[0].size
        assert all(im.size == nbytes for im in imgs)
        ptrs = (c_u8p * n)(*[_p(im, c_u8p) for im in imgs])
        out = np.zeros(imgs[0].shape, np.uint8)
        self._ck(self.L.cgrt_average_u8(self.h, n, ptrs, C.c_int64(nbytes), _p(out, c_u8p)))
        return out

    def average_f64(self, images, want_rgb8=False):
        imgs = [_d(im) for im in images]
        n, nv = len(imgs), imgs[0].size
        assert all(im.size == nv for im in imgs)
        ptrs = (c_dp * n)(*[_p(im, c_dp) for im in imgs])
        mean = np.zeros(imgs[0].shape)
        rgb8 = np.zeros(imgs[0].shape, np.uint8) if want_rgb8 else None
        self._ck(self.L.cgrt_average_f64(self.h, n, ptrs, C.c_int64(nv), _p(mean, c_dp), _p(rgb8, c_u8p)))
        return (mean, rgb8) if want_rgb8 else mean

    # -- downloads
    def num_hitpoints(self):
        n = C.c_int64(0)
        self._ck(self.L.cgrt_num_hitpoints(self.h, C.byref(n)))
        return n.value

    def download_hitpoints(self, fields=None):
        """Canonical order. `fields`: subset of the keys to fetch (default all) — the others are passed as NULL."""
        n = self.num_hitpoints()
        spec = dict(pos=((n, 3), np.float64), normal=((n, 3), np.float64), f=((n, 3), np.float64), flux=((n, 3), np.float64), r2=((n,), np.float64),
                    n=((n,), np.int32), hw=((n, 2), np.int32), key=((n,), np.uint32), seq=((n,), np.uint32))
        o = {k: np.zeros(sh, dt) for k, (sh, dt) in spec.items() if fields is None or k in fields}
        g = o.get
        self._ck(self.L.cgrt_download_hitpoints(self.h, _p(g("pos"), c_dp), _p(g("normal"), c_dp), _p(g("f"), c_dp), _p(g("flux"), c_dp), _p(g("r2"), c_dp),
                                                _p(g("n"), c_ip), _p(g("hw"), c_ip), _p(g("key"), c_up), _p(g("seq"), c_up)))
        return o

    def download_accum(self):
        n = self.num_hitpoints()
        df = np.zeros((n, 3)); m = np.zeros(n)
        self._ck(self.L.cgrt_download_accum(self.h, _p(df, c_dp), _p(m, c_dp)))
        return df, m

    def download_grid(self):
        cs = np.zeros(self.cfg.hashsize + 1, np.uint32)
        self._ck(self.L.cgrt_download_grid(self.h, _p(cs, c_up)))
        return cs

    def counters(self):
        k = CgrtCounters()
        self._ck(self.L.cgrt_get_counters(self.h, C.byref(k)))
        return {n: int(getattr(k, n)) for n, _ in CgrtCounters._fields_}

    def set_counting(self, on=True):
        self._ck(self.L.cgrt_set_counting(self.h, int(on)))

    def set_culling(self, on=True):
        self._ck(self.L.cgrt_set_culling(self.h, int(on)))

    def set_overlap(self, on=True):
        self._ck(self.L.cgrt_set_overlap(self.h, int(on)))

    def check_guards(self) -> int:
        """Damaged fence bytes so far (only meaningful when the process was started with CGRT_GUARD=1)."""
        n = C.c_uint64(0)
        self._ck(self.L.cgrt_check_guards(self.h, C.byref(n)))
        return int(n.value)

    @staticmethod
    def release_cached_memory(device=-1) -> int:
        """cudaFree the large buffers the library parked for later contexts (-1: every device). -> bytes released"""
        n = C.c_uint64(0)
        load_library().cgrt_release_cached_memory(int(device), C.byref(n))
        return int(n.value)

    def photon_chunk(self) -> int:
        n = C.c_uint64(0)
        self._ck(self.L.cgrt_photon_chunk(self.h, C.byref(n)))
        return int(n.value)

    # -- multi-GPU through the C ABI (NCCL bound at run time)
    def set_comm(self, comm, world):
        self._ck(self.L.cgrt_set_comm(self.h, C.c_void_p(comm), int(world)))

    def allgather_hitpoints(self, comm, world):
        self._ck(self.L.cgrt_allgather_hitpoints(self.h, C.c_void_p(comm), int(world)))

    def allreduce_accum(self, comm):
        self._ck(self.L.cgrt_allreduce_accum(self.h, C.c_void_p(comm)))

    def peer_export(self) -> bytes:
        """This rank's 128-byte handle of its accumulator block (after build_grid); see cgrt_peer_export."""
        buf = C.create_string_buffer(128)
        self._ck(self.L.cgrt_peer_export(self.h, buf))
        return buf.raw

    def peer_attach(self, rank: int, world: int, handles) -> None:
        """handles: the `world` blobs of peer_export in rank order. From now on round_update exchanges over peer memory."""
        blob = b"".join(handles)
        assert len(blob) == 128 * world
        self._ck(self.L.cgrt_peer_attach(self.h, int(rank), int(world), blob))

    def set_profiling(self, on=True):
        self._ck(self.L.cgrt_set_profiling(self.h, int(on)))

    def timings(self):
        ms = (C.c_double * 12)()
        self._ck(self.L.cgrt_get_timings(self.h, ms))
        names = ["eye", "grid", "photon_trace", "photon_deposit", "update", "gather", "deposit_sort", "trace_traverse", "trace_continue",
                 "trace_emit", "allgather", "r11"]
        return {n: ms[i] for i, n in enumerate(names)}


def comm_unique_id() -> bytes:
    """128-byte ncclUniqueId (make it on rank 0, hand it to every rank)."""
    buf = C.create_string_buffer(128)
    rc = load_library().cgrt_comm_unique_id(buf)
    if rc != 0:
        raise CgrtError(f"cgrt_comm_unique_id failed with status {rc} (is NCCL loadable?)")
    return buf.raw


def comm_init_rank(device: int, rank: int, world: int, uid: bytes) -> int:
    """-> ncclComm_t as an integer handle (collective: every rank must call it)."""
    comm = C.c_void_p()
    rc = load_library().cgrt_comm_init_rank(int(device), int(rank), int(world), C.c_char_p(uid), C.byref(comm))
    if rc != 0:
        raise CgrtError(f"cgrt_comm_init_rank failed with status {rc}")
    return comm.value


def comm_destroy(comm: int) -> None:
    load_library().cgrt_comm_destroy(C.c_void_p(comm))
