"""propagate_normal_orientations (SURVEY.md §8f rank 4) without a GPU: the oracle's sequential
restatement against fixtures produced by the UNMODIFIED reference with its own kd-tree
(tests/golden/ref_orient.npz) and against the live reference bridge when present.  Signs are
bit-exact: the normals are only ever negated."""
import os

import numpy as np
import pytest

FIX = os.path.join(os.path.dirname(__file__), "golden", "ref_orient.npz")
CASES = ["sphere", "random", "blobs"]


@pytest.fixture(scope="module")
def fix():
    return np.load(FIX)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_fixture(oracle, fix, name):
    xyz, nrm, k = fix[name + "_xyz"], fix[name + "_normals"], int(fix[name + "_k"])
    idx, _, _ = oracle.cloud(xyz).knn(None, k)
    out = oracle.propagate_normal_orientations(xyz, idx, nrm, reverse_edges=True)
    assert np.array_equal(out, fix[name + "_oriented"])
    root = int(np.argmax(xyz[:, 2]))
    assert np.array_equal(out[root], np.array([0, 0, 1], np.float32))
    others = np.arange(len(xyz)) != root
    assert np.array_equal(np.abs(out[others]), np.abs(nrm[others]))  # only ever negated


def test_sphere_becomes_consistent(fix):
    xyz, out = fix["sphere_xyz"], fix["sphere_oriented"]
    radial = xyz / np.linalg.norm(xyz, axis=1, keepdims=True)
    assert ((out * radial).sum(1) > 0).all()  # root is the north pole, (0,0,1) points outward


def test_unreached_component_keeps_normals(fix):
    xyz, nrm, out = fix["blobs_xyz"], fix["blobs_normals"], fix["blobs_oriented"]
    root = int(np.argmax(xyz[:, 2]))
    assert root < 1500
    assert np.array_equal(out[1500:], nrm[1500:])


def test_edge_order_matters_and_libstdcxx_is_reverse(oracle, fix):
    xyz, nrm, k = fix["random_xyz"], fix["random_normals"], int(fix["random_k"])
    idx, _, _ = oracle.cloud(xyz).knn(None, k)
    fwd = oracle.propagate_normal_orientations(xyz, idx, nrm, reverse_edges=False)
    assert not np.array_equal(fwd, fix["random_oriented"])


def test_oracle_matches_live_reference(oracle):
    from oracle_lib import RefOrient, have_ref_orient

    if not have_ref_orient():
        pytest.skip("oracle/_ref/libpcp_ref_orient.so not built (set PCP_REFERENCE to a reference "
                    "checkout)")
    ref = RefOrient()
    rng = np.random.default_rng(6)
    xyz = np.stack([rng.uniform(0, 1, 3000), rng.uniform(0, 1, 3000),
                    0.02 * rng.standard_normal(3000)], 1).astype(np.float32)
    nrm = rng.standard_normal((3000, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    for k in (1, 4, 12):
        idx, _, _ = oracle.cloud(xyz).knn(None, k)
        mine = oracle.propagate_normal_orientations(xyz, idx, nrm)
        assert np.array_equal(mine, ref.propagate_normal_orientations(xyz, k, nrm, knn=idx))
        assert np.array_equal(mine, ref.propagate_normal_orientations(xyz, k, nrm))
