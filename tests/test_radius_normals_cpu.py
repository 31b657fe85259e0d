"""The ball PCA (pcpx_estimate_normals_radius) without a GPU: the checker against numpy brute
force, and the device body (radius_normal in normals_core.cuh, run on the host by the
emulation library) against the checker.  Counts bit-exact; normals 1 - |cos| <= 1e-4 where the
eigengap > 1e-3; centroids within 1e-5 * max(1, max|p|) of the fp64 mean of the exact ball."""
import numpy as np
import pytest

from ball_oracle import (bruteforce_ball_normals, centroid_tolerance, normal_error,
                         radius_normals)


@pytest.fixture(scope="module")
def ball_emu():
    from emu_ball_lib import BallEmu

    return BallEmu()


def check_against(xyz, got_nrm, got_ctr, got_cnt, want_nrm, gap, want_ctr, want_cnt):
    assert np.array_equal(got_cnt, want_cnt)
    well = gap > 1e-3
    if well.any():
        assert normal_error(got_nrm, want_nrm)[well].max() <= 1e-4
    full = want_cnt > 0
    assert np.isnan(got_ctr[~full]).all()
    if full.any():
        assert np.abs(got_ctr[full] - want_ctr[full]).max() <= centroid_tolerance(xyz)
    assert (got_nrm[~full] == np.float32([0, 0, 1])).all()


def emu_vs_oracle(ball_emu, oracle, xyz, queries, r, radii=None, bbox=None, min_well=0.0):
    ix, oc = ball_emu.index(xyz, bbox=bbox), oracle.cloud(xyz, bbox=bbox)
    nrm, ctr, cnt = ix.radius_normals(queries, r, radii)
    onrm, octr, gap, ocnt = radius_normals(oc, queries, r, radii)
    assert np.array_equal(cnt, ix.radius_count(queries, r, radii))
    check_against(xyz, nrm, ctr, cnt, onrm, gap, octr, ocnt)
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1, atol=1e-5)
    assert (gap > 1e-3).mean() >= min_well
    return nrm, ctr, cnt, gap


def test_oracle_against_numpy_bruteforce(oracle, pcpx):
    xyz = pcpx.synth.noisy_sphere(4000, seed=3)
    rng = np.random.default_rng(0)
    q = np.concatenate([xyz[rng.choice(len(xyz), 300, replace=False)],
                        rng.uniform(-1.2, 1.2, (100, 3)).astype(np.float32)])
    oc = oracle.cloud(xyz)
    for r in (0.05, 0.12):
        onrm, octr, gap, ocnt = radius_normals(oc, q, r)
        bnrm, bctr, bgap, bcnt = bruteforce_ball_normals(xyz, q, r)
        assert np.array_equal(ocnt, bcnt)
        assert (bcnt > 0).mean() > 0.7
        check_against(xyz, onrm, octr, ocnt, bnrm, bgap, bctr, bcnt)
        assert np.abs(gap - bgap).max() < 1e-3


@pytest.mark.parametrize("shape", ["plane", "sphere", "noise_mix"])
def test_emulated_body_on_surfaces(ball_emu, oracle, pcpx, shape):
    if shape == "plane":
        xyz, r = pcpx.synth.noisy_plane(6000, extent=1.0, sigma=1e-3), 0.04
    elif shape == "sphere":
        xyz, r = pcpx.synth.noisy_sphere(6000), 0.12
    else:
        xyz, r = pcpx.synth.noise_mix(6000, extent=1.0), 0.04
    rng = np.random.default_rng(1)
    ext = (xyz[rng.choice(len(xyz), 500)] + rng.normal(0, 0.01, (500, 3))).astype(np.float32)
    far = np.float32([[50, 50, 50]])
    emu_vs_oracle(ball_emu, oracle, xyz, None, r, min_well=0.9)
    emu_vs_oracle(ball_emu, oracle, xyz, np.concatenate([ext, far]), r)
    # against the fp64 brute force as well (the centroid tolerance is defined on it)
    nrm, ctr, cnt = ball_emu.index(xyz).radius_normals(ext[:150], r)
    bnrm, bctr, bgap, bcnt = bruteforce_ball_normals(xyz, ext[:150], r)
    check_against(xyz, nrm, ctr, cnt, bnrm, bgap, bctr, bcnt)


def test_lattice_points_exactly_at_r_are_in_the_ball(ball_emu, oracle):
    # spacing 1/8 in x, y and 1/4 between layers: every in-layer neighbour at distance exactly r
    g = np.arange(12, dtype=np.float32) * np.float32(0.125)
    x, y, z = np.meshgrid(g, g, np.arange(3, dtype=np.float32) * np.float32(0.25), indexing="ij")
    xyz = np.stack([x.ravel(), y.ravel(), z.ravel()], 1).astype(np.float32)
    nrm, ctr, cnt, gap = emu_vs_oracle(ball_emu, oracle, xyz, None, 0.125)
    inner = ((xyz[:, 0] > 0) & (xyz[:, 0] < g[-1]) & (xyz[:, 1] > 0) & (xyz[:, 1] < g[-1]))
    assert (cnt[inner] == 5).all()  # itself + 4 neighbours at exactly r
    assert np.array_equal(ctr[inner], xyz[inner])  # symmetric ball
    assert (np.abs(nrm[inner, 2]) == 1).all()


def test_duplicates(ball_emu, oracle):
    rng = np.random.default_rng(5)
    base = rng.uniform(0, 1, (1500, 3)).astype(np.float32)
    base[:, 2] *= np.float32(0.01)
    xyz = np.concatenate([base, base, base[:500]], 0)
    emu_vs_oracle(ball_emu, oracle, xyz, None, 0.06)
    # r = 0: a ball of identical points has zero scatter -> (0,0,1) exactly
    nrm, ctr, cnt = ball_emu.index(xyz).radius_normals(None, 0.0)
    assert (cnt >= 2).all()
    assert (nrm == np.float32([0, 0, 1])).all()
    assert np.array_equal(ctr, xyz)


def test_per_query_radii_including_zero(ball_emu, oracle, pcpx):
    xyz = pcpx.synth.noisy_plane(5000, extent=1.0)
    rng = np.random.default_rng(9)
    q = np.concatenate([xyz[:300], rng.uniform(0, 1, (200, 3)).astype(np.float32)])
    radii = rng.uniform(0, 0.08, len(q)).astype(np.float32)
    radii[::7] = 0
    nrm, ctr, cnt, _ = emu_vs_oracle(ball_emu, oracle, xyz, q, 123.0, radii=radii)
    assert (cnt[:300][radii[:300] == 0] == 1).all()  # the point itself
    one = cnt == 1
    assert (nrm[one] == np.float32([0, 0, 1])).all()
    assert np.array_equal(ctr[:300][radii[:300] == 0], q[:300][radii[:300] == 0])
    emu_vs_oracle(ball_emu, oracle, xyz, None, 0.0, radii=rng.uniform(0, 0.06, len(xyz)))


def test_voxel_grid_leaves_points_out_of_every_ball(ball_emu, oracle):
    rng = np.random.default_rng(6)
    xyz = rng.uniform(-2, 2, (5000, 3)).astype(np.float32)
    xyz[:, 2] *= np.float32(0.05)
    box = np.array([-1, -1, -1, 1, 1, 1], np.float32)
    nrm, ctr, cnt, _ = emu_vs_oracle(ball_emu, oracle, xyz, None, 0.2, bbox=box)
    inside = (np.abs(xyz) <= 1).all(1)
    assert 0 < inside.sum() < len(xyz)
    # every query, indexed or not, sees exactly the indexed points of its ball
    bnrm, bctr, bgap, bcnt = bruteforce_ball_normals(xyz[inside], xyz, 0.2)
    check_against(xyz, nrm, ctr, cnt, bnrm, bgap, bctr, bcnt)
    assert (cnt[~inside] == 0).any() and (cnt[inside] >= 1).all()


def test_offset_cloud_keeps_its_accuracy(ball_emu, oracle, pcpx):
    xyz = (pcpx.synth.noisy_plane(4000, extent=1.0).astype(np.float64) + 1000.0).astype(np.float32)
    nrm, ctr, cnt = ball_emu.index(xyz).radius_normals(xyz[:400], 0.05)
    bnrm, bctr, bgap, bcnt = bruteforce_ball_normals(xyz, xyz[:400], 0.05)
    check_against(xyz, nrm, ctr, cnt, bnrm, bgap, bctr, bcnt)
    assert (bgap > 1e-3).mean() > 0.9
