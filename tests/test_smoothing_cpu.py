"""Radius-search callers (SURVEY.md §8f rank 3) without a GPU: the oracle's restatement of the
bilateral filter and WLOP is pinned against (i) fixtures produced by the UNMODIFIED reference
(tests/golden/ref_smoothing.npz, made by make_smoothing_fixtures.py), (ii) the live reference
bridge when oracle/_ref is present and (iii) the reference's own test expectations; then the
device code (smoothing_core.cuh compiled for the host by tests/emu) is compared with the oracle.

All of this is fp32 with a data-dependent summation order (the reference sums neighbours in
kd-tree order, the oracle in octree order, the index in cell order), so the tolerance is
absolute: 2e-5 of the cloud's extent for positions, 1 - |cos| <= 1e-5 for normals."""
import os

import numpy as np
import pytest

from golden import kats

FIX = os.path.join(os.path.dirname(__file__), "golden", "ref_smoothing.npz")
POS_TOL = 2e-5  # x cloud extent


@pytest.fixture(scope="module")
def fix():
    return np.load(FIX)


def close(a, b, extent):
    return float(np.abs(a.astype(np.float64) - b).max()) <= POS_TOL * extent


def extent_of(xyz):
    return float((xyz.max(0) - xyz.min(0)).max())


# ---- oracle <-> reference ---------------------------------------------------------------------
def test_oracle_bilateral_line_kat(oracle, fix):
    pts, nrm = kats.BILATERAL_LINE_POINTS, kats.BILATERAL_LINE_NORMALS
    sigmaf = float(oracle.cloud(pts).mean_knn_distance(kats.BILATERAL_LINE_KNN)[1])
    assert abs(sigmaf - float(fix["line_sigmaf"])) < 1e-7
    out = oracle.bilateral_filter_points(pts, nrm, sigmaf, sigmaf / 8.0, kats.BILATERAL_LINE_K)
    # test/algorithm/bilateral_filter.cpp:121-125
    assert pts[2, 2] > out[2, 2] and pts[6, 2] < out[6, 2]
    assert close(out, fix["line_points"], 0.2)


def test_oracle_bilateral_matches_reference_fixture(oracle, fix):
    xyz, nrm = fix["shell_xyz"], fix["shell_normals"]
    for it in (1, 3):
        out = oracle.bilateral_filter_points(xyz, nrm, 0.08, 0.02, it)
        assert close(out, fix["shell_bilateral_K%d" % it], extent_of(xyz))


def test_oracle_wlop_matches_reference_fixture(oracle, fix):
    xyz, init = fix["shell_xyz"], fix["shell_wlop_initial"]
    for uniform in (1, 0):
        out = oracle.wlop(xyz, init, 0.45, 0.15, 3, bool(uniform))
        assert close(out, fix["shell_wlop_uniform%d" % uniform], extent_of(xyz))
    cube = kats.wlop_case() * kats.WLOP_PARITY_SCALE
    out = oracle.wlop(cube, fix["cube_wlop_initial"], 0.45, float(fix["cube_h"]), 2, True)
    assert close(out, fix["cube_wlop"], extent_of(cube))
    # test/algorithm/wlop.cpp:53-88 at its own scale: I points, none NaN / Inf
    cube = kats.wlop_case()
    h = float(oracle.cloud(cube).mean_knn_distance(15)[1])
    out = oracle.wlop(cube, fix["cube_wlop_initial"], 0.45, h, 2, True)
    assert out.shape == (len(cube) // 2, 3) and np.isfinite(out).all()


def test_oracle_matches_live_reference(oracle):
    from oracle_lib import RefSmoothing, have_ref_smoothing

    if not have_ref_smoothing():
        pytest.skip("oracle/_ref/libpcp_ref_smoothing.so not built (set PCP_REFERENCE to a reference "
                    "checkout)")
    ref = RefSmoothing()
    rng = np.random.default_rng(77)
    xyz = np.stack([rng.uniform(0, 1, 2500), rng.uniform(0, 1, 2500),
                    0.01 * rng.standard_normal(2500)], 1).astype(np.float32)
    nrm = np.tile(np.array([0, 0, 1], np.float32), (2500, 1))
    nrm += 0.2 * rng.standard_normal(nrm.shape).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    a = oracle.bilateral_filter_points(xyz, nrm, 0.04, 0.01, 2)
    assert close(a, ref.bilateral_filter_points(xyz, nrm, 0.04, 0.01, 2), 1.0)
    init = rng.permutation(2500)[:600].astype(np.uint32)
    for uniform in (True, False):
        a = oracle.wlop(xyz, init, 0.3, 0.08, 4, uniform)
        assert close(a, ref.wlop(xyz, init, 0.3, 0.08, 4, uniform), 1.0)


def test_oracle_bilateral_normals_properties(oracle, fix):
    # unpinned by the reference (its test only checks the count, bilateral_filter.cpp:135-155):
    # unit length and K = 0 is the identity.  (The map is NOT translation invariant: :243 builds
    # the Jacobian of the numerator from s_projected - s but :204 / :250 use the absolute
    # s_projected; restated as written.)
    xyz, nrm = fix["shell_xyz"][:1500], fix["shell_normals"][:1500]
    out = oracle.bilateral_filter_normals(xyz, nrm, 0.1, 0.025, 2)
    assert out.shape == nrm.shape
    assert np.allclose(np.linalg.norm(out, axis=1), 1.0, atol=1e-5)
    assert np.array_equal(oracle.bilateral_filter_normals(xyz, nrm, 0.1, 0.025, 0), nrm)


# ---- device code (host build) <-> oracle ------------------------------------------------------
def test_emu_bilateral_points(emu, oracle, fix):
    pts, nrm = kats.BILATERAL_LINE_POINTS, kats.BILATERAL_LINE_NORMALS
    s = float(fix["line_sigmaf"])
    assert close(emu.bilateral_filter_points(pts, nrm, s, s / 8, 2), fix["line_points"], 0.2)
    xyz, nrm = fix["shell_xyz"], fix["shell_normals"]
    for it in (1, 3):
        out = emu.bilateral_filter_points(xyz, nrm, 0.08, 0.02, it)
        assert close(out, fix["shell_bilateral_K%d" % it], extent_of(xyz))
        assert close(out, oracle.bilateral_filter_points(xyz, nrm, 0.08, 0.02, it),
                     extent_of(xyz))


def test_emu_bilateral_normals(emu, oracle, fix):
    xyz, nrm = fix["shell_xyz"], fix["shell_normals"]
    for it in (1, 2):
        a = emu.bilateral_filter_normals(xyz, nrm, 0.08, 0.02, it)
        b = oracle.bilateral_filter_normals(xyz, nrm, 0.08, 0.02, it)
        assert float((1 - np.abs((a * b).sum(1))).max()) <= 1e-5
        assert float(((a * b).sum(1)).min()) > 0  # same sign too: the map is not sign-free


def test_emu_wlop(emu, oracle, fix):
    xyz, init = fix["shell_xyz"], fix["shell_wlop_initial"]
    for uniform in (1, 0):
        out = emu.wlop(xyz, init, 0.45, 0.15, 3, bool(uniform))
        assert close(out, fix["shell_wlop_uniform%d" % uniform], extent_of(xyz))
    cube = kats.wlop_case() * kats.WLOP_PARITY_SCALE
    out = emu.wlop(cube, fix["cube_wlop_initial"], 0.45, float(fix["cube_h"]), 2, True)
    assert np.isfinite(out).all() and close(out, fix["cube_wlop"], extent_of(cube))
    cube = kats.wlop_case()  # the reference test's own scale: exact ball, I finite points
    out = emu.wlop(cube, fix["cube_wlop_initial"], 0.45, 2.5, 2, True)
    assert out.shape == (len(cube) // 2, 3) and np.isfinite(out).all()
    assert close(out, oracle.wlop(cube, fix["cube_wlop_initial"], 0.45, 2.5, 2, True),
                 extent_of(cube))
    # no neighbours at all (h far below the spacing): every point stays where it is
    out = emu.wlop(cube, fix["cube_wlop_initial"], 0.45, 1e-4, 2, True)
    assert np.array_equal(out, cube[fix["cube_wlop_initial"]])
    assert np.array_equal(out, oracle.wlop(cube, fix["cube_wlop_initial"], 0.45, 1e-4, 2, True))
