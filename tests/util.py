import numpy as np


def random_rays(n, seed=0, inside_room=True):
    """Rays with origins inside the 40x40x50 room and isotropic directions (the photon-like incoherent case)."""
    rng = np.random.default_rng(seed)
    o = rng.uniform(-19.5, 19.5, (n, 3))
    o[:, 2] = rng.uniform(-9.0, 39.5, n)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1)[:, None]
    return np.ascontiguousarray(o), np.ascontiguousarray(d)


def camera_rays(width, height, step=1):
    """main.cpp:188-198 pinhole rays through pixel corners."""
    hs, ws = np.meshgrid(np.arange(0, height, step), np.arange(0, width, step), indexing="ij")
    x = (2.0 * (ws.astype(np.float64) / width) - 1) * 10.0
    y = (2.0 * (hs.astype(np.float64) / height) - 1) * 10.0 * height / width
    d = np.stack([x, y, np.zeros_like(x)], -1).reshape(-1, 3) - np.array([0, 0, -10.0])
    nrm = np.sqrt(d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1] + d[:, 2] * d[:, 2])
    d = d * (1 / nrm)[:, None]
    o = np.tile(np.array([[0, 0, -10.0]]), (len(d), 1))
    return np.ascontiguousarray(o), np.ascontiguousarray(d)


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), 1e-300)


def assert_flux_close(df, odf, om, accum):
    """Per-hitpoint flux accumulators of the GPU (df) against the oracle's (odf, fp64), om = accepted photons per hitpoint.
    accum 0 (fp64 atomics): only the order of the additions differs -> 1e-9 relative.
    accum 1 (float `red` accumulators): every deposit is positive, so summing m of them in float in ANY order is within
    (m - 1 + roundings of one term) * 2^-24 of the exact sum, relative — the worst-case bound of recursive summation."""
    err = np.abs(np.asarray(df, np.float64) - odf)
    if accum == 0:
        assert np.all(err <= 1e-9 * np.abs(odf) + 1e-9), float(err.max())
    else:
        bound = (np.asarray(om, np.float64)[:, None] + 8.0) * 2.0 ** -24 * np.abs(odf) + 1e-6
        assert np.all(err <= bound), float((err / bound).max())
        pos = odf > 0
        assert np.median(err[pos] / odf[pos]) < 5e-7  # and typically a few ulp


class OracleEngine:
    """The engine protocol of cgraytracing_b200.distributed.ShardedRenderer over the CPU oracle. `sppm` (the oracle's SPPM mode, 0: PPM)
    tells ShardedRenderer whether to call eye_pass once or sppm_eye_pass every round."""

    def __init__(self, scene, cfg, sppm=0):
        from oracle import binding as ob

        self.o = ob.Oracle(scene, cfg)
        self.sppm = sppm
        if sppm:
            self.o.set_sppm(sppm)

    def eye_pass(self, y0, y1):
        self.o.eye_pass(y0, y1)

    def sppm_eye_pass(self, r, y0, y1):
        self.o.sppm_eye_pass(r, y0, y1)

    def export_hitpoints(self):
        import torch

        return torch.from_numpy(self.o.export_hitpoints())

    def import_hitpoints(self, rec):
        self.o.import_hitpoints(rec.numpy())

    def build_grid(self):
        self.o.build_grid()

    def photon_pass(self, first, count):
        self.o.photon_pass(first, count)

    def accum_tensor(self):
        import torch

        df, m = self.o.download_accum()
        return torch.from_numpy(np.concatenate([df, m[:, None].astype(np.float64)], 1).copy())

    def accum_commit(self, t):
        a = t.numpy()
        self.o.upload_accum(a[:, :3], a[:, 3].astype(np.int32))

    def round_update(self):
        self.o.round_update()

    def gather_image(self, n):
        return self.o.gather_image(n)
