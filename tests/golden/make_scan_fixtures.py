"""Generates tests/golden/ref_scans.npz: the reference's real scans
($PCP_REFERENCE/examples/data/{stanford_bunny,fandisk,detergent,spray}.ply, SURVEY.md §8c) read
by the UNMODIFIED reference PLY reader and pushed through the UNMODIFIED reference octree and
kd-tree (oracle/_ref/libpcp_ref*.so): full-cloud kNN k = 15 (indices + squared distances),
sphere-range counts at r = 2 x the mean 15-NN distance, per-point mean 15-NN distance.  The
clouds themselves are stored too (the scans are not part of this repository).  Only runnable
with PCP_REFERENCE naming a reference checkout.

    PCP_REFERENCE=<checkout> python tests/golden/make_scan_fixtures.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle_lib import REFERENCE_DIR, RefBridge, RefPly  # noqa: E402

DATA = os.path.join(REFERENCE_DIR or "$PCP_REFERENCE", "examples", "data")
SCANS = ["stanford_bunny", "fandisk", "detergent", "spray"]


def main():
    ply, ref = RefPly(), RefBridge()
    out = {}
    for name in SCANS:
        xyz, _ = ply.read(open(os.path.join(DATA, name + ".ply"), "rb").read())
        assert len(xyz) > 1000, (name, len(xyz))
        rc = ref.cloud(xyz)
        idx, d2, cnt = rc.knn(0, None, 15)
        idx2, d22, _ = rc.knn(1, None, 15)
        assert np.array_equal(idx, idx2) and np.array_equal(d2, d22), name  # octree == kd-tree
        means, mu = rc.mean_knn_distance(0, 15)
        r = np.float32(min(1.0, 2.0 * float(mu)))
        off, _ = rc.radius_search(0, None, r)
        off2, _ = rc.radius_search(1, None, r)
        assert np.array_equal(off, off2), name
        out[name + "_xyz"] = xyz
        out[name + "_k15_idx"] = idx.astype(np.int32)
        out[name + "_k15_d2"] = d2
        out[name + "_mean15"] = means
        out[name + "_radius_r"] = r
        out[name + "_radius_count"] = np.diff(off.astype(np.int64)).astype(np.uint32)
        print(name, len(xyz), "points, mean 15-NN distance", float(mu), "mean ball count",
              float(out[name + "_radius_count"].mean()))
    path = os.path.join(HERE, "ref_scans.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
