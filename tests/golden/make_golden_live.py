#!/usr/bin/env python
"""Generates tests/golden/ref_live.npz: the cases of tests/test_ref_live_golden.py (the live comparisons of tests/test_oracle_vs_ref.py
and tests/test_mirror.py) as digests and sampled rows of their outputs.

    python tests/golden/make_golden_live.py            # from the compiled reference (make -C oracle REF=<reference checkout>)
    python tests/golden/make_golden_live.py oracle     # from the CPU oracle, where the reference is not available

The fixture records which side wrote it in `source`. One written from the oracle holds the reference's outputs only as far as the
oracle is bit-exact to the reference on these inputs, which tests/test_oracle_vs_ref.py checks; on a machine with the reference,
tests/test_ref_live_golden.py::test_stored_outputs_equal_the_live_reference checks the fixture itself.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import binding as ob  # noqa: E402
from tests.test_ref_live_golden import CASES, GOLDEN, fixture_entries  # noqa: E402


def main(side):
    if side == "ref":
        assert ob.have_ref(), "build oracle/_ref first: make -C oracle REF=<reference checkout>"
    ob.build()
    g = {"source": np.array("compiled reference (oracle/_ref/libcgref.so)" if side == "ref" else "CPU oracle (oracle/ppm_oracle.hpp)")}
    for name, case in CASES.items():
        g.update(fixture_entries(name, *case(ob, side)))
    np.savez_compressed(GOLDEN, **g)
    print("wrote", GOLDEN, os.path.getsize(GOLDEN), "bytes,", len(g), "arrays, source:", g["source"])


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "ref")
