"""ctypes wrapper of tests/sppm_split_oracle.cpp: the SPPM CPU reference (tests/sppm_oracle.cpp) with the round split the way ranks of several
GPUs run it — a row tile of the eye pass into a pending set, the record exchange, then the table. TEST INFRASTRUCTURE ONLY.

Compiled once per process into a temporary directory with the flags of tests/sppm_oracle.py. Everything SppmOracle offers works as well."""
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from tests.sppm_oracle import CXXFLAGS, SppmOracle, _d, _p, c_dp, c_ip

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "sppm_split_oracle.cpp")

_lib = None


def lib():
    global _lib
    if _lib is None:
        out_dir = tempfile.mkdtemp(prefix="sppm_split_oracle_")
        so = os.path.join(out_dir, "libsppm_split_oracle.so")
        env = dict(os.environ)
        env.pop("CXX", None)
        env.pop("CC", None)
        subprocess.check_call([shutil.which("g++") or "g++"] + CXXFLAGS + ["-o", so, SRC], env=env)
        L = C.CDLL(so)
        L.sppm_create.restype = C.c_void_p
        L.sppm_destroy.argtypes = [C.c_void_p]
        L.sppm_num_visible.restype = C.c_int64
        L.sppm_num_visible.argtypes = [C.c_void_p]
        L.sppm_pending_create.restype = C.c_void_p
        L.sppm_pending_destroy.argtypes = [C.c_void_p]
        L.sppm_export_pending.restype = C.c_int64
        _lib = L
    return _lib


class SppmSplitOracle(SppmOracle):
    """SppmOracle plus the split round: eye_rows(r, y0, y1) -> export_pending / import_pending -> build_table -> photon_pass ->
    (download_hitpoints, all-reduce, upload_accum) -> round_update."""

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
        self.pending = C.c_void_p(self.L.sppm_pending_create())
        self.cfg = cfg
        scene.build_into(self)

    def close(self):
        if getattr(self, "pending", None):
            self.L.sppm_pending_destroy(self.pending)
            self.pending = None
        super().close()

    def eye_rows(self, r, y0=0, y1=-1, nthreads=1):
        """Round r's eye pass over rows [y0, y1) into the pending set; the table is not built."""
        assert self.L.sppm_eye_rows(self.h, self.pending, C.c_uint32(r), int(y0), int(y1), int(nthreads)) == 0

    def export_pending(self):
        """-> float64 [n, 12] records of the pending visible points (the format of oracle.binding.Oracle.export_hitpoints)."""
        n = int(self.L.sppm_export_pending(self.h, self.pending, None))
        rec = np.zeros((n, 12))
        if n:
            self.L.sppm_export_pending(self.h, self.pending, _p(rec, c_dp))
        return rec

    def import_pending(self, rec):
        rec = _d(rec).reshape(-1, 12)
        assert self.L.sppm_import_pending(self.h, self.pending, C.c_int64(len(rec)), _p(rec, c_dp)) == 0

    def build_table(self):
        """The pending visible points into the round's table, canonical order, each at its pixel's radius."""
        assert self.L.sppm_build_table(self.h, self.pending) == 0

    def upload_accum(self, dflux, m):
        df = _d(dflux).reshape(-1, 3)
        mm = np.ascontiguousarray(m, dtype=np.int32)
        assert self.L.sppm_upload_accum(self.h, _p(df, c_dp), _p(mm, c_ip)) == 0
