"""Helpers of tests/test_fixed_accum.py: the fixed-point oracle behind ShardedRenderer's engine protocol, and renders that return every
observable of a finished render (n, r2, flux, linear image, rgb8)."""
import numpy as np

from tests.util import OracleEngine


class FixedOracleEngine(OracleEngine):
    """OracleEngine over oracle_fixed.FixedOracle: the accumulator tensor is the int64 {sum q, M} block, all-reduced exactly."""

    def __init__(self, scene, cfg, sppm=0, nthreads=1):
        from oracle_fixed.binding import FixedOracle

        self.o = FixedOracle(scene, cfg)
        self.sppm = sppm
        self.nthreads = nthreads
        if sppm:
            self.o.set_sppm(sppm)

    def photon_pass(self, first, count):
        self.o.photon_pass(first, count, self.nthreads)

    def accum_tensor(self):
        import torch

        return torch.from_numpy(self.o.download_accum_i64())

    def accum_commit(self, t):
        self.o.upload_accum_i64(t.numpy())


def observables(ctx_or_oracle, sppm, n_emitted, rgb8=None):
    """n, r2, flux (PPM: per hitpoint; SPPM: per pixel, tau) and the linear image of a context or oracle after its last round_update."""
    img = ctx_or_oracle.gather_image(n_emitted)
    if sppm:
        p = ctx_or_oracle.sppm_download_pixels()
        out = dict(n=p["n"], r2=p["r2"], flux=p["tau"], img=img)
    else:
        h = ctx_or_oracle.download_hitpoints(fields=("n", "r2", "flux", "pos", "key"))
        out = dict(n=h["n"], r2=h["r2"], flux=h["flux"], pos=h["pos"], key=h["key"], img=img)
    if rgb8 is not None:
        out["rgb8"] = rgb8
    return out


def assert_same(a, b, keys=None):
    for k in keys or sorted(set(a) & set(b)):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
