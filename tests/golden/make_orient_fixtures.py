"""Generates tests/golden/ref_orient.npz by running the UNMODIFIED reference's
propagate_normal_orientations (oracle/_ref/libpcp_ref_orient.so) with its own kd-tree kNN on
small seeded clouds.  Only runnable with PCP_REFERENCE naming a reference checkout; the
committed .npz travels.

    PCP_REFERENCE=<checkout> python tests/golden/make_orient_fixtures.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle_lib import RefOrient  # noqa: E402


def cases():
    rng = np.random.default_rng(404)
    d = rng.standard_normal((4000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sphere = (d * (1 + 0.005 * rng.standard_normal((4000, 1)))).astype(np.float32)
    flip = np.where(rng.uniform(size=(4000, 1)) < 0.5, -1.0, 1.0)
    yield "sphere", sphere, (d * flip).astype(np.float32), 10  # true normals, random signs
    r = rng.standard_normal((4000, 3))
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    yield "random", sphere, r.astype(np.float32), 6  # every sign depends on the BFS tree
    # two well separated blobs: the second one is never reached and keeps its normals
    blob = rng.uniform(0, 1, (1500, 3))
    two = np.concatenate([blob, blob * 0.5 + [5, 5, -3]], 0).astype(np.float32)
    r2 = rng.standard_normal((3000, 3))
    r2 /= np.linalg.norm(r2, axis=1, keepdims=True)
    yield "blobs", two, r2.astype(np.float32), 8


def main():
    ref = RefOrient()
    out = {}
    for name, xyz, nrm, k in cases():
        out[name + "_xyz"], out[name + "_normals"], out[name + "_k"] = xyz, nrm, np.int64(k)
        out[name + "_oriented"] = ref.propagate_normal_orientations(xyz, k, nrm)
    path = os.path.join(HERE, "ref_orient.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
