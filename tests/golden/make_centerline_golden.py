"""Generates tests/golden/centerline_rca_short.npz. Run with a checkout of the reference:

    python tests/golden/make_centerline_golden.py <reference checkout>

The reference's example RCA centerline (examples/data/centerline_rca_short.csv, 788 x [x, y, z]; five concatenated
vessel segments) re-encoded so the branch tests of tests/test_intravascular.py:249-343 can run without the
reference."""
import sys
from pathlib import Path

import numpy as np

src = Path(sys.argv[1]) / "examples/data/centerline_rca_short.csv"
xyz = np.genfromtxt(src, delimiter=",")
assert xyz.shape == (788, 3), xyz.shape
np.savez_compressed(Path(__file__).resolve().parent / "centerline_rca_short.npz", xyz=xyz)
print("wrote", xyz.shape)
