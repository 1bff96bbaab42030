"""Generates tests/golden/golden_mill1024_v1.json: CRC32 of the two raybuffers for 6 poses of the benchmark path on
datasets/mill.obj at 1024^3, 1920x1080 (the cases of test_mill_1024_matches_the_translated_reference_1080p), so that the test
has its expected values without the reference's library.

Where oracle/_ref can be built (oracle/ref.py) the vectors come from it and the oracle must agree with every one of them;
otherwise they come from the oracle (oracle/cpuvox_oracle.cpp), which reproduces the reference's vectors of
tests/golden/golden_ref_v1.json. The file's "generator" names the source.
    python tests/golden/make_golden_mill1024.py
"""
from __future__ import annotations

import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cpuvox_b200 as cv  # noqa: E402  (host side only: world builder, pose helpers, segment setup)
from conftest import MILL, crc  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from oracle import ref  # noqa: E402

W, H = 1920, 1080
POSE_INDICES = (0, 12, 24, 36, 48, 59)


def main():
    world = cv.World.from_obj(MILL, 1024)
    lods = cv.setup_lods(world.max_dimension, W, H)
    poses = cv.benchmark_path(world.dims, 60, far_clip=2.0 * world.max_dimension)
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rw = ref.RefWorld(world.dims, world.blobs, world.column_counts) if ref.build() else None
    cases = {}
    for i in POSE_INDICES:
        s = cv.frame_setup(poses[i], W, H, lods, world.dims[1])
        td, lr, _ = orc.render_raybuffers(ow, orc.copy_setup(s), W, H)
        if rw is not None:
            rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H)
            assert (td == rtd).all() and (lr == rlr).all(), f"the oracle differs from the reference at pose {i}"
        cases[str(i)] = [crc(td), crc(lr)]
    out = {"version": 1, "generator": ref.describe() if rw is not None else "oracle/cpuvox_oracle.cpp",
           "world": "datasets/mill.obj at 1024^3", "width": W, "height": H,
           "blob_crcs": [crc(b) for b in world.blobs], "cases": cases}
    with open(os.path.join(ROOT, "tests", "golden", "golden_mill1024_v1.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
