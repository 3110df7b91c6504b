"""Two ranks of a multi-GPU SPPM render emulated by contexts of ONE device (test infrastructure of tests/test_sppm_multi_gpu.py).

Each context plays a rank: it traces its row tile of the round's eye pass (cgrt_sppm_eye_pass), the records of all tiles are concatenated
in rank order with torch and imported into every context (what cgrt_allgather_hitpoints does over NCCL), every context builds the grid and
traces its photon range, and the accumulators are summed with torch and written back into every context before cgrt_round_update (what
the all-reduce inside cgrt_round_update does). Everything of the library's multi-GPU SPPM path runs except the NCCL calls themselves.

Run as a script (with CGRT_GUARD=1 in the environment) it drives the emulation with fenced device buffers and reports the damaged fence
bytes:  CGRT_GUARD=1 python tests/sppm_two_ranks.py
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _dev(ptr, n, typestr):
    import torch

    from cgraytracing_b200.distributed import _DevArray

    return torch.as_tensor(_DevArray(ptr, n, typestr), device="cuda:0")


def sppm_context(cg, scene, cfg, mode, accum):
    g = cg.Context(0)
    g.set_config(cfg, accum_mode=accum)
    scene.build_into(g)
    g.commit()
    g.set_sppm(mode)
    return g


def emulated_round(ranks, r, nph, height, on_grid=None):
    """Round r over the contexts in `ranks` (rank order). on_grid(ranks) runs after every rank has built the round's grid."""
    import torch

    from cgraytracing_b200.distributed import HP_RECORD_DOUBLES, photon_shard, row_shard

    world = len(ranks)
    for k, g in enumerate(ranks):
        y0, y1 = row_shard(height, k, world)
        g.sppm_eye_pass(r, y0, y1)
    parts = []
    for g in ranks:
        ptr, n = g.export_hitpoints_dev()
        if n:
            parts.append(_dev(ptr, n * HP_RECORD_DOUBLES, "<f8").view(n, HP_RECORD_DOUBLES))
    union = torch.cat(parts, 0) if parts else torch.zeros((0, HP_RECORD_DOUBLES), dtype=torch.float64, device="cuda:0")
    torch.cuda.synchronize()
    for g in ranks:
        g.import_hitpoints_dev(union.data_ptr(), union.shape[0])
    for g in ranks:
        g.build_grid()
    if on_grid is not None:
        on_grid(ranks)
    for k, g in enumerate(ranks):
        first, count = photon_shard(r, nph, k, world)
        if count:
            g.photon_pass(first, count)
    for g in ranks:
        g.synchronize()
    accs = []
    for g in ranks:
        ptr, n = g.accum_dev()
        accs.append(_dev(ptr, n, "<f8" if g.accum_mode == 0 else "<f4") if n else None)
    if accs[0] is not None:
        total = accs[0].clone()
        for a in accs[1:]:
            total += a
        for a in accs:
            a.copy_(total)
        torch.cuda.synchronize()
    for g in ranks:
        g.round_update()


GUARD_CASES = (("c3_dragon_glass", 20000, dict(width=64, height=64), 30000),
               ("c4_bump_dof", None, dict(width=64, height=36, use_dof=1, num_of_samples=2), 30000))


def guard_probe():
    import numpy as np

    import cgraytracing_b200 as cg

    damaged = 0
    for name, max_tris, kw, P in GUARD_CASES:
        s = cg.preset(name, max_tris=max_tris)
        cfg = cg.RenderConfig(**kw)
        for mode, accum in ((1, 0), (1, 1), (2, 1)):
            ranks = [sppm_context(cg, s, cfg, mode, accum) for _ in range(2)]
            try:
                for r in range(3):
                    emulated_round(ranks, r, P, cfg.height)
                img = ranks[0].gather_image(3.0 * P)
                n = ranks[0].sppm_download_pixels()["n"]
                damaged += sum(g.check_guards() for g in ranks)
            finally:
                for g in ranks:
                    g.close()
            print(f"{name:16s} mode {mode} accum {accum}: pixels with photons {int((n > 0).sum())} mean {img.mean():.4f} "
                  f"finite {bool(np.isfinite(img).all())}", flush=True)
    print("probe done; guard mode", os.environ.get("CGRT_GUARD", "0"), "damaged fence bytes", damaged)
    return damaged


if __name__ == "__main__":
    sys.exit(1 if guard_probe() else 0)
