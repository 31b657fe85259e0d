"""Generates tests/golden/ref_smoothing.npz by running the UNMODIFIED reference
(oracle/_ref/libpcp_ref_smoothing.so: pcp::algorithm::bilateral_filter_points and the
pcp::algorithm::wlop::detail bodies, compiled in place from $PCP_REFERENCE/include) on small
seeded clouds.  Only runnable with PCP_REFERENCE naming a reference checkout; the committed
.npz travels.

    PCP_REFERENCE=<checkout> python tests/golden/make_smoothing_fixtures.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import kats  # noqa: E402
from oracle_lib import RefBridge, RefSmoothing  # noqa: E402


def shell(n, seed):
    rng = np.random.default_rng(seed)
    d = rng.standard_normal((n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    xyz = (d * (1 + 0.01 * rng.standard_normal((n, 1)))).astype(np.float32)
    nrm = d + 0.1 * rng.standard_normal((n, 3))
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    return xyz, nrm.astype(np.float32)


def main():
    ref, tree = RefSmoothing(), RefBridge()
    out = {}
    # the reference's own bilateral test: sigmaf from its kd-tree (test/.../bilateral_filter.cpp:85-101)
    pts, nrm = kats.BILATERAL_LINE_POINTS, kats.BILATERAL_LINE_NORMALS
    sigmaf = float(tree.cloud(pts).mean_knn_distance(1, kats.BILATERAL_LINE_KNN)[1])
    out["line_sigmaf"] = np.float64(sigmaf)
    out["line_points"] = ref.bilateral_filter_points(pts, nrm, sigmaf, sigmaf / 8.0,
                                                     kats.BILATERAL_LINE_K)
    xyz, nrm = shell(3000, 31)
    out["shell_xyz"], out["shell_normals"] = xyz, nrm
    for it in (1, 3):
        out["shell_bilateral_K%d" % it] = ref.bilateral_filter_points(xyz, nrm, 0.08, 0.02, it)
    rng = np.random.default_rng(8)
    init = rng.permutation(len(xyz))[:750].astype(np.uint32)
    out["shell_wlop_initial"] = init
    for uniform in (1, 0):
        out["shell_wlop_uniform%d" % uniform] = ref.wlop(xyz, init, 0.45, 0.15, 3, bool(uniform))
    cube = kats.wlop_case() * kats.WLOP_PARITY_SCALE
    h = float(tree.cloud(cube).mean_knn_distance(1, 15)[1])
    init = np.random.default_rng(9).permutation(len(cube))[:len(cube) // 2].astype(np.uint32)
    out["cube_h"] = np.float64(h)
    out["cube_wlop_initial"] = init
    out["cube_wlop"] = ref.wlop(cube, init, 0.45, h, 2, True)
    path = os.path.join(HERE, "ref_smoothing.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes;", len(out), "arrays")


if __name__ == "__main__":
    main()
