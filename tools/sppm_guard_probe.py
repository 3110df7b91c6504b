"""SPPM rounds of every BASELINE scene family through the C ABI with fenced device buffers (CGRT_GUARD=1): every buffer of a context sits
between two 4 KiB fences, and the probe fails when a kernel has written into one. Covers the per-round release and re-allocation of the
visible points and the grid, the fold kernel and the pixel image, for both camera modes and both accumulator types.
tests/test_sppm.py runs it.

  CGRT_GUARD=1 python tools/sppm_guard_probe.py
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cgraytracing_b200 import Context, RenderConfig, preset  # noqa: E402

CASES = (("c1_spheres_bezier", dict(width=48, height=48), 20000),
         ("c2_bunny_chess", dict(width=64, height=64), 30000),
         ("c3_dragon_glass", dict(width=64, height=64), 30000),
         ("c4_bump_dof", dict(width=64, height=36, use_dof=1, num_of_samples=2), 30000))
damaged = 0
for name, kw, P in CASES:
    s = preset(name)
    for mode, accum in ((1, 0), (1, 1), (2, 1)):
        with Context(0) as g:
            g.set_config(RenderConfig(**kw), accum_mode=accum)
            s.build_into(g); g.commit()
            g.set_sppm(mode)
            for r in range(3):
                g.sppm_begin_round(r)
                g.photon_pass(r * P, P); g.round_update()
            img, rgb8 = g.gather_image(3.0 * P, want_rgb8=True)
            px = g.sppm_download_pixels()
            c = g.counters()
            damaged += g.check_guards()
            print(f"{name:18s} mode {mode} accum {accum}: visible points {c['hitpoints']} deposits {c['deposits']} pixels with photons "
                  f"{int((px['n'] > 0).sum())} mean {img.mean():.4f} finite {bool(np.isfinite(img).all())}", flush=True)
print("probe done; guard mode", os.environ.get("CGRT_GUARD", "0"), "damaged fence bytes", damaged)
sys.exit(1 if damaged else 0)
