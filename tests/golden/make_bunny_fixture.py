"""Writes tests/golden/bun10k_points.npz: the vertex payload of the reference's benchmark cloud.

The reference's benchmark and notebook load examples/data/bun10k.ply (reference benchmarks/main.cpp:156-167,
examples/python/ex4_bunny.ipynb) -- binary little-endian PLY, 235-byte header, 9992 vertices of float32 x, y, z
(SURVEY.md section 8c row 4).  The project does not ship the reference tree, so the INPUT vectors travel as this small
fixture (119 904 bytes of float32, stored losslessly), written by this script from a checkout of the reference.
tests/test_oracle_golden.py::test_bunny_fixture_matches_ply pins the fixture to the SHA-256 of that vertex payload.

usage:  python tests/golden/make_bunny_fixture.py <reference checkout>/examples/data/bun10k.ply"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from clipper_b200 import datagen  # noqa: E402

if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__.splitlines()[-1])
    xyz = datagen.read_ply_xyz(sys.argv[1])
    assert xyz.shape == (9992, 3) and xyz.dtype == np.float32
    np.savez_compressed(os.path.join(HERE, "bun10k_points.npz"), xyz=xyz)
    print("bun10k_points.npz:", xyz.shape, xyz.dtype, "extent", xyz.max(0) - xyz.min(0))
