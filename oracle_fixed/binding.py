"""ctypes binding of the CPU oracle with fixed-point accumulators (oracle_fixed/libfxorc.so). TEST INFRASTRUCTURE ONLY.

FixedOracle is an oracle.binding.Oracle (the library contains the whole oracle C API) whose photon pass, round update and accumulator
downloads use the fixed-point definition of accum_mode 2 (include/cgrt.h)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from oracle.binding import Oracle, _d, _p, c_dp

HERE = os.path.dirname(os.path.abspath(__file__))
FX_SO = os.path.join(HERE, "libfxorc.so")
_SOURCES = (os.path.join(HERE, "fixed_capi.cpp"), os.path.join(HERE, "..", "oracle", "oracle_capi.cpp"),
            os.path.join(HERE, "..", "oracle", "ppm_oracle.hpp"))
c_i64p = C.POINTER(C.c_int64)
c_fp = C.POINTER(C.c_float)

ERR_VALUE, ERR_COUNT = 1, 2

_fx = None


def build(force: bool = False) -> None:
    if force or not os.path.exists(FX_SO) or os.path.getmtime(FX_SO) < max(os.path.getmtime(f) for f in _SOURCES):
        subprocess.check_call(["make", "-C", HERE, "-s"])


def fx_lib():
    global _fx
    if _fx is None:
        build()
        L = C.CDLL(FX_SO)
        L.fxo_create.restype = C.c_void_p
        L.fxo_destroy.argtypes = [C.c_void_p]
        L.orc_num_hitpoints.restype = C.c_int64
        L.orc_num_hitpoints.argtypes = [C.c_void_p]
        L.orc_texture_height.restype = C.c_double
        L.orc_texture_height.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.orc_hash.restype = C.c_uint32
        _fx = L
    return _fx


class FixedOracle(Oracle):
    """The oracle in the fixed-point mode: photon_pass deposits q = round-half-even(cf * 2^22), round_update reads sum q * 2^-22."""

    def __init__(self, scene=None, config=None):
        self.L = fx_lib()
        self.h = C.c_void_p(self.L.fxo_create())
        self.cfg = None
        if config is not None:
            self.set_config(config)
        if scene is not None:
            scene.build_into(self)

    def close(self):
        if self.h:
            self.L.fxo_destroy(self.h)
            self.h = None

    def photon_pass(self, first, count, nthreads=1, reverse=False):
        r = self.L.fxo_photon_pass(self.h, C.c_uint64(first), C.c_uint64(count), int(nthreads), int(bool(reverse)))
        assert r == 0, r

    def trace(self, org, dir, flux, adj=None, flag=False, x=0, y=0, path=0):
        """A caller-made photon (flag must be False) with fixed-point deposits."""
        assert not flag, "the fixed-point mode changes only the photon side"
        r = self.L.fxo_trace(self.h, _p(_d(org), c_dp), _p(_d(dir), c_dp), _p(_d(flux), c_dp), C.c_uint64(path))
        assert r == 0, r

    def round_update(self):
        assert self.L.fxo_round_update(self.h) == 0

    def download_accum(self):
        """-> (sum q * 2^-22 [n, 3], M [n]) as float64, like Context.download_accum in accum_mode 2."""
        n = self.num_hitpoints()
        df = np.zeros((n, 3)); m = np.zeros(n)
        self.L.fxo_download_accum(self.h, None, _p(df, c_dp), _p(m, c_dp))
        return df, m

    def download_accum_i64(self):
        """-> int64 [n, 4] {sum q_x, sum q_y, sum q_z, M} in canonical order."""
        a = np.zeros((self.num_hitpoints(), 4), np.int64)
        self.L.fxo_download_accum(self.h, _p(a, c_i64p), None, None)
        return a

    def upload_accum_i64(self, acc4):
        a = np.ascontiguousarray(acc4, dtype=np.int64).reshape(-1, 4)
        assert len(a) == self.num_hitpoints()
        self.L.fxo_upload_accum(self.h, _p(a, c_i64p))

    def error(self):
        """ERR_VALUE | ERR_COUNT bits raised so far."""
        return int(self.L.fxo_error(self.h))


def deposit_value(f, flux):
    """The definition on free-standing inputs: -> (cf float32, q int64) per element of f * flux."""
    f = np.ascontiguousarray(f, dtype=np.float64).ravel()
    flux = np.ascontiguousarray(np.broadcast_to(flux, f.shape), dtype=np.float64).ravel()
    cf = np.zeros(f.shape, np.float32); q = np.zeros(f.shape, np.int64)
    fx_lib().fxo_deposit_value(C.c_int64(len(f)), _p(f, c_dp), _p(flux, c_dp), _p(cf, c_fp), _p(q, c_i64p))
    return cf, q
