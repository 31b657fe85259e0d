"""Generates tests/golden/ref_fixtures.npz by running the UNMODIFIED reference (through
oracle/_ref/libpcp_ref.so, i.e. $PCP_REFERENCE/include compiled in place) on small seeded
clouds.  Only runnable with PCP_REFERENCE naming a reference checkout; the committed .npz is
what travels.

    PCP_REFERENCE=<checkout> python tests/golden/make_fixtures.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle_lib import RefBridge  # noqa: E402


def clouds():
    rng = np.random.default_rng(2024)
    d = rng.standard_normal((3000, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sphere = (d * (1 + 0.005 * rng.standard_normal((3000, 1)))).astype(np.float32)
    cube = rng.uniform(-100, 100, (2500, 3)).astype(np.float32)
    plane = np.stack([rng.uniform(0, 1, 3000), rng.uniform(0, 1, 3000),
                      1e-3 * rng.standard_normal(3000)], 1).astype(np.float32)
    # duplicates and near-duplicates (inside the 1e-5 exclusion box), lattice ties
    g = np.stack(np.meshgrid(*[np.arange(8)] * 3, indexing="ij"), -1).reshape(-1, 3)
    lattice = (g * 0.125).astype(np.float32)
    dup = np.concatenate([plane[:500], plane[:500] + np.float32(3e-6), plane[:200]], 0)
    return {"sphere": sphere, "cube": cube, "plane": plane, "lattice": lattice, "dup": dup}


def main():
    ref = RefBridge()
    out = {}
    rng = np.random.default_rng(99)
    for name, xyz in clouds().items():
        rc = ref.cloud(xyz)
        ext = xyz.max(0) - xyz.min(0)
        q = (xyz.min(0) - 0.1 * ext + rng.uniform(0, 1, (400, 3)) * 1.2 * ext).astype(np.float32)
        out[name + "_xyz"] = xyz
        out[name + "_queries"] = q
        # the reference's octree and kd-tree must agree (tie-aware order); one copy is stored
        for k in (1, 8, 15):
            for qq, qn in ((None, "self"), (q, "ext")):
                idx, d2, cnt = rc.knn(0, qq, k)
                idx2, d22, cnt2 = rc.knn(1, qq, k)
                assert np.array_equal(idx, idx2) and np.array_equal(d2, d22), (name, k, qn)
                out["%s_%s_k%d_idx" % (name, qn, k)] = idx.astype(np.int32)
                out["%s_%s_k%d_d2" % (name, qn, k)] = d2
        scale = float(ext.max())
        for frac, lists in ((0.02, True), (0.1, False)):
            r = np.float32(min(1.0, frac * scale))  # parity contract: r <= 1 (SURVEY.md §3.3)
            off, ids = rc.radius_search(0, None, r)
            off2, ids2 = rc.radius_search(1, None, r)
            assert np.array_equal(off, off2) and np.array_equal(ids, ids2), (name, frac)
            out["%s_radius_%g_count" % (name, frac)] = np.diff(off.astype(np.int64)).astype(np.uint32)
            if lists:
                out["%s_radius_%g_idx" % (name, frac)] = ids.astype(np.int32)
            out["%s_radius_%g_r" % (name, frac)] = r
            cq = rc.radius_count(0, q, r)
            assert np.array_equal(cq, rc.radius_count(1, q, r))
            out["%s_radius_%g_ext_count" % (name, frac)] = cq
        means, mu = rc.mean_knn_distance(0, 15)
        out[name + "_mean15"] = means
        out[name + "_mean15_mu"] = mu
    np.savez_compressed(os.path.join(HERE, "ref_fixtures.npz"), **out)
    print("wrote", os.path.join(HERE, "ref_fixtures.npz"), len(out), "arrays")


if __name__ == "__main__":
    main()
