"""Generates tests/golden/ref_ply.npz: the byte streams the UNMODIFIED reference writer
(pcp::io::write_ply, through oracle/_ref/libpcp_ref_ply.so) produces for a small cloud in each
of the three formats.  Only runnable with PCP_REFERENCE naming a reference checkout; the .npz
travels.

    PCP_REFERENCE=<checkout> python tests/golden/make_ply_fixtures.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle_lib import RefPly  # noqa: E402


def main():
    ref = RefPly()
    rng = np.random.default_rng(55)
    xyz = (rng.standard_normal((257, 3)) * [1, 10, 1e-3]).astype(np.float32)
    xyz[0] = (0.0, -0.0, 1.0)
    xyz[1] = (1e-7, 123456.789, -3.5)  # std::to_string's fixed six decimals
    nrm = rng.standard_normal((257, 3))
    nrm = (nrm / np.linalg.norm(nrm, axis=1, keepdims=True)).astype(np.float32)
    out = {"xyz": xyz, "normals": nrm}
    for fmt in RefPly.FORMATS:
        out[fmt] = np.frombuffer(ref.write(xyz, nrm, fmt), np.uint8)
        out[fmt + "_no_normals"] = np.frombuffer(ref.write(xyz, nrm[:0], fmt), np.uint8)
    path = os.path.join(HERE, "ref_ply.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
