"""Rigid registration (pcpx_nearest_within, pcpx_icp) without a GPU: the device bodies
(icp_core.cuh) and the host solve (icp_solve.hpp), run on the host by the emulation library,
against numpy: the bounded nearest neighbour index for index and bit for bit against a kd-tree
brute force, the normal equations against fp64 numpy sums, the solver against numpy's eigh
pseudo-inverse and SVD Kabsch.  The C++ program (tests/cpp/icp_test.cpp) is compiled with strict
warnings here and run on the GPU by tests/test_gpu_icp.py."""
import os

import numpy as np
import pytest

from emu_icp_lib import (NONE, brute_nearest_within, np_solve, np_step, np_sums, np_update,
                         pose_error, rigid, transform_f32)

F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz")
SCANS = os.path.join(ROOT, "tests", "golden", "ref_scans.npz")
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]


@pytest.fixture(scope="module")
def icp_emu():
    from emu_icp_lib import IcpEmu

    return IcpEmu()


def _cloud(name):
    if name in CLOUDS:
        return np.load(FIX)[name + "_xyz"].astype(F32)
    return np.load(SCANS)[name + "_xyz"].astype(F32)


def _extent(xyz):
    return float(np.linalg.norm(xyz.max(0).astype(np.float64) - xyz.min(0)))


def check_nearest(icp_emu, target, queries, r, T=None, voxel_grid=None):
    target = np.asarray(target, F32).reshape(-1, 3)
    indexed = None
    if voxel_grid is not None:
        lo, hi = (np.asarray(v, F32) for v in voxel_grid)
        indexed = np.all((target >= lo) & (target <= hi), axis=1)
    with icp_emu.index(target, voxel_grid) as ix:
        got_i, got_d = ix.nearest_within(queries, r, T)
    y = queries if T is None else transform_f32(queries, T)
    want_i, want_d = brute_nearest_within(target, y, r, indexed)
    assert np.array_equal(got_i, want_i), np.nonzero(got_i != want_i)[0][:10]
    assert np.array_equal(got_d.view(np.uint32), want_d.view(np.uint32))
    return got_i, got_d


@pytest.mark.parametrize("name", CLOUDS + SCAN_NAMES)
def test_nearest_within_reference_clouds(icp_emu, name):
    xyz = _cloud(name)
    ext = _extent(xyz)
    rng = np.random.default_rng(1)
    q = xyz[rng.integers(0, len(xyz), 3000)] + rng.normal(0, 0.01 * ext, (3000, 3)).astype(F32)
    T = rigid(4.0, [1, 2, 3], 0.01 * ext * np.array([1, -1, 0.5]))
    for r in (0.005 * ext, 0.03 * ext, 2.0 * ext):
        check_nearest(icp_emu, xyz, q, r)
        check_nearest(icp_emu, xyz, q, r, T)
    # the cloud's own points: d2 0 at themselves (or an earlier duplicate)
    got, d2 = check_nearest(icp_emu, xyz, xyz, 0.01 * ext)
    assert (d2 == 0).all()


def test_nearest_within_exact_tie_lattice(icp_emu):
    g = np.arange(8, dtype=F32)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    # queries at cell centres, face centres and edge midpoints: 8, 4 and 2 equidistant points
    q = np.concatenate([xyz[:200] + F32(0.5), xyz[:200] + np.array([0.5, 0.5, 0], F32),
                        xyz[:200] + np.array([0.5, 0, 0], F32)])
    for r in (0.5, 0.8660254, 0.9, 3.0):
        got, _ = check_nearest(icp_emu, xyz, q, r)
    assert (got != NONE).all()


def test_nearest_within_bound_is_inclusive(icp_emu):
    # a line spaced exactly r: the neighbour at d2 == fl(r * r) is in; one float below it is out
    r = F32(0.25)
    xyz = np.zeros((64, 3), F32)
    xyz[:, 0] = np.arange(64, dtype=F32) * r
    q = xyz[:32] + np.array([r / 2, 0, 0], F32)  # halfway: the lower index wins the tie
    got, _ = check_nearest(icp_emu, xyz[::2], xyz[1::2], r)
    assert (got[:-1] != NONE).all()
    below = np.nextafter(r, F32(0))
    got, _ = check_nearest(icp_emu, xyz[::2], xyz[1::2], below)
    assert (got == NONE).all()
    got, _ = check_nearest(icp_emu, xyz, q, r)
    assert np.array_equal(got, np.arange(32))


def test_nearest_within_outside_nan_voxel_grid_offset(icp_emu):
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0, 1, (20000, 3)).astype(F32)
    far = rng.uniform(-1, 2, (4000, 3)).astype(F32)  # many outside the root voxel
    check_nearest(icp_emu, xyz, far, 0.05)
    check_nearest(icp_emu, xyz, far, 0.6)
    nan = far[:50].copy()
    nan[::3, 0] = np.nan
    nan[1::3, 1] = np.inf
    got, d2 = check_nearest(icp_emu, xyz, nan, 10.0)
    assert (got[::3] == NONE).all() and np.isinf(d2[1::3]).all()
    vox = (np.array([0.2, 0.2, 0.2], F32), np.array([0.7, 0.8, 0.9], F32))
    check_nearest(icp_emu, xyz, far, 0.1, voxel_grid=vox)
    off = xyz + F32(1000)
    check_nearest(icp_emu, off, far + F32(1000), 0.05)
    check_nearest(icp_emu, off, xyz + F32(1000), 0.02, rigid(3, [0, 0, 1], [0.01, 0, 0]))


def test_nearest_within_empty_index(icp_emu):
    got, d2 = icp_emu.index(np.zeros((0, 3), F32)).nearest_within(np.ones((5, 3), F32), 1.0)
    assert (got == NONE).all() and np.isinf(d2).all()


def _plane_normals(xyz, k=10):
    from scipy.spatial import cKDTree

    _, nb = cKDTree(xyz).query(xyz, k=k)
    P = xyz[nb].astype(np.float64)
    P -= P.mean(1, keepdims=True)
    _, V = np.linalg.eigh(np.einsum("nki,nkj->nij", P, P))
    return V[:, :, 0].astype(F32)


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("name", ["stanford_bunny", "fandisk"])
def test_normal_equations(icp_emu, name, metric):
    xyz = _cloud(name)
    ext = _extent(xyz)
    nrm = _plane_normals(xyz)
    nrm[::97] = np.nan  # pairs with such a normal are no pairs (point-to-plane)
    T = rigid(5, [0, 1, 1], 0.01 * ext * np.ones(3))
    with icp_emu.index(xyz) as ix:
        s, corr = ix.sums(xyz, 0.05 * ext, metric, T, nrm)
        _, want = np_step(metric, xyz, nrm, xyz, 0.05 * ext, T, ix.centre)
    assert s[-1] == want[-1] and s[-1] > 100
    assert np.allclose(s, want, rtol=1e-12, atol=1e-12 * np.abs(want).max())
    y = transform_f32(xyz, T)
    bi, _ = brute_nearest_within(xyz, y, 0.05 * ext)
    if metric == 0:
        bad = (bi != NONE) & ~np.all(np.isfinite(nrm[np.minimum(bi, len(xyz) - 1)]), axis=1)
        bi[bad] = NONE
    assert np.array_equal(corr, bi)


def test_solver_matches_numpy(icp_emu):
    rng = np.random.default_rng(7)
    for _ in range(20):
        J = rng.normal(size=(200, 6))
        r = rng.normal(size=200)
        A = J.T @ J
        s = np.concatenate([A[np.triu_indices(6)], J.T @ r, [1.0, 200]])
        x = icp_emu.solve(0, s)
        assert np.allclose(x, np_solve(0, s), rtol=1e-12, atol=1e-12 * np.abs(x).max())
        y = rng.normal(size=(50, 3))
        R = rigid(rng.uniform(1, 170), rng.normal(size=3), rng.normal(size=3))
        q = (R[:3, :3] @ y.T).T + R[:3, 3] + 1e-3 * rng.normal(size=(50, 3))
        c = rng.normal(size=3)
        s = np_sums(1, y.astype(F32), q.astype(F32), np.zeros(50), c)
        x = icp_emu.solve(1, s)
        assert np.allclose(x, np_solve(1, s), rtol=1e-10, atol=1e-12)
        T = rng.normal(size=(4, 4))
        T[3] = [0, 0, 0, 1]
        assert np.allclose(icp_emu.update(T, x, c), np_update(T, x, c), rtol=1e-12, atol=1e-12)


def test_solver_rank_deficient_plane(icp_emu):
    # a plane z = 0 registered to itself shifted by dz and tilted: the in-plane translations and
    # the rotation about the normal are unconstrained, and must come out exactly zero
    rng = np.random.default_rng(11)
    q = np.c_[rng.uniform(-1, 1, (500, 2)), np.zeros(500)]
    n = np.tile([0.0, 0.0, 1.0], (500, 1))
    y = q.copy()
    y[:, 2] = 0.01 + 0.02 * y[:, 0]
    s = np_sums(0, y.astype(F32), q.astype(F32), np.zeros(500), np.zeros(3), n.astype(F32))
    x = icp_emu.solve(0, s)
    assert np.allclose(x, np_solve(0, s), rtol=1e-12, atol=1e-14)
    assert x[2] == 0 and x[3] == 0 and x[4] == 0
    assert abs(x[5] + 0.01) < 1e-6 and abs(x[1] - 0.02) < 1e-6


@pytest.mark.parametrize("metric", [0, 1])
def test_emulated_icp_recovers_a_motion(icp_emu, metric):
    xyz = _cloud("stanford_bunny")
    ext = _extent(xyz)
    nrm = _plane_normals(xyz)
    M = rigid(6, [1, -2, 1], 0.015 * ext * np.array([1, 0.5, -1]))
    src = transform_f32(xyz, M)
    with icp_emu.index(xyz) as ix:
        T, (its, stop, pairs), corr = ix.icp(src, 0.1 * ext, metric, nrm, max_it=60)
        assert stop == 0 and pairs > 0.95 * len(xyz)
        ang, dist = pose_error(T, np.linalg.inv(M))
        assert ang < 1e-5 and dist < 1e-5 * ext
        # one step equals the numpy step from the same start
        T1, (its1, _, _), _ = ix.icp(src, 0.1 * ext, metric, nrm, max_it=1)
        W, _ = np_step(metric, xyz, nrm, src, 0.1 * ext, np.eye(4), ix.centre)
        assert its1 == 1
        assert np.abs(T1[:3, :3] - W[:3, :3]).max() < 1e-9
        assert np.abs(T1[:3, 3] - W[:3, 3]).max() < 1e-9 * ext


def test_emulated_icp_stops(icp_emu):
    xyz = _cloud("fandisk")
    with icp_emu.index(xyz) as ix:
        _, (its, stop, pairs), corr = ix.icp(xyz[:2], 1.0, 1)
        assert (its, stop, pairs) == (0, 2, 2)
        _, (its, stop, _), _ = ix.icp(xyz + F32(0.001), 1.0, 1, max_it=2, rot_tol=1e-30,
                                       trans_tol=1e-30)
        assert (its, stop) == (2, 1)
