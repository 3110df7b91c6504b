"""Worker of tests/test_bvh_edges.py: one photon round of c3 (20,000 triangles), run in a process of its own because the library reads
CGRT_TRAV_EXACT (force the fp64-slab traversal of photons) once per process. Writes the accepted counts, flux and counters to argv[1]."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

W, H, NPH = 64, 48, 20000


def main():
    from cgraytracing_b200 import Context, RenderConfig, preset

    cfg = RenderConfig(width=W, height=H, into_rule=1, update_mode=1)
    with Context(0, preset("c3_dragon_glass", max_tris=20000), cfg) as g:
        g.eye_pass(); g.build_grid()
        g.photon_pass(0, NPH)
        df, m = g.download_accum()
        k = g.counters()
    names = sorted(k)
    np.savez(sys.argv[1], df=df, m=m, names=np.array(names), counters=np.array([k[n] for n in names], np.uint64))


if __name__ == "__main__":
    main()
