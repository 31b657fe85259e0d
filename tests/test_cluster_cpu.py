"""Density-based clustering (pcpx_cluster_by_density) without a GPU: the device bodies
(cluster_core.cuh, run on the host by the emulation library with a sequential union-find) against
a brute-force DBSCAN of the same contract (tests/emu_cluster_lib.py: bruteforce_dbscan), label for
label.  The checker itself is pinned on a hand-labelled cloud."""
import numpy as np
import pytest

from emu_cluster_lib import NOISE, bruteforce_dbscan

F32 = np.float32
ROOT_GOLDEN = "tests/golden"
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]


@pytest.fixture(scope="module")
def cluster_emu():
    from emu_cluster_lib import ClusterEmu

    return ClusterEmu()


def _golden(name):
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    return np.load(os.path.join(root, ROOT_GOLDEN, name))


def check(cluster_emu, xyz, r, min_points, voxel_grid=None):
    """emulated labels == brute force, label for label; returns (labels, n_clusters, core)"""
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    indexed = None
    if voxel_grid is not None:
        lo, hi = (np.asarray(v, F32) for v in voxel_grid)
        indexed = np.all((xyz >= lo) & (xyz <= hi), axis=1)
    got, nc, core = cluster_emu.cluster(xyz, r, min_points, voxel_grid)
    want, wnc, wcore = bruteforce_dbscan(xyz, r, min_points, indexed)
    assert np.array_equal(core, wcore)
    assert nc == wnc
    assert np.array_equal(got, want), np.nonzero(got != want)[0][:10]
    # numbering: 0 .. C-1, first appearance among core points in ascending index order
    seen = got[core]
    if len(seen):
        _, first = np.unique(seen, return_index=True)
        assert np.array_equal(seen[np.sort(first)], np.arange(nc))
    return got, nc, core


def test_checker_on_a_hand_labelled_cloud():
    # blob A (indices 0-3) around x = 0, blob B (4-7) around x = 3, r = 1, min_points 4: every
    # blob point is core.  Point 9 at x = 1.5 has 3 points in its ball: it is a border point at
    # d2 == 1 from blob A's point 1 and from blob B's point 5, and the tie goes to the lower
    # index.  Points 8 and 10 are within reach of nothing: noise.
    xyz = np.array([[0, 0, 0], [0.5, 0, 0], [0, 0.5, 0], [0, 0, 0.5],
                    [3, 0, 0], [2.5, 0, 0], [3, 0.5, 0], [3, 0, 0.5],
                    [1.5, 5, 0], [1.5, 0, 0], [40, 40, 40]], F32)
    labels, nc, core = bruteforce_dbscan(xyz, 1.0, 4)
    assert core.tolist() == [True] * 8 + [False] * 3
    assert nc == 2
    assert labels.tolist() == [0, 0, 0, 0, 1, 1, 1, 1, NOISE, 0, NOISE]
    # the same cloud listed with blob B first: B is cluster 0, and the tie still goes to the
    # lower index, now B's point
    perm = [4, 5, 6, 7, 0, 1, 2, 3, 8, 9, 10]
    labels, nc, _ = bruteforce_dbscan(xyz[perm], 1.0, 4)
    assert labels.tolist() == [0, 0, 0, 0, 1, 1, 1, 1, NOISE, 0, NOISE]
    # min_points 1: every point is core; the middle point joins both blobs into one cluster
    labels, nc, core = bruteforce_dbscan(xyz, 1.0, 1)
    assert core.all() and nc == 3
    assert labels.tolist() == [0] * 8 + [1, 0, 2]


def test_hand_labelled_cloud(cluster_emu):
    xyz = np.array([[0, 0, 0], [0.5, 0, 0], [0, 0.5, 0], [0, 0, 0.5],
                    [3, 0, 0], [2.5, 0, 0], [3, 0.5, 0], [3, 0, 0.5],
                    [1.5, 5, 0], [1.5, 0, 0], [40, 40, 40]], F32)
    for mp in (0, 1, 3, 4, 5):
        check(cluster_emu, xyz, 1.0, mp)
    labels, nc, _ = cluster_emu.cluster(xyz, 1.0, 4)
    assert nc == 2 and labels.tolist() == [0, 0, 0, 0, 1, 1, 1, 1, NOISE, 0, NOISE]


@pytest.mark.parametrize("name", CLOUDS)
@pytest.mark.parametrize("min_points", [1, 5, 15])
def test_reference_fixture_clouds(cluster_emu, name, min_points):
    z = _golden("ref_fixtures.npz")
    xyz = z[name + "_xyz"]
    for tag in ("0.02", "0.1"):
        r = z["%s_radius_%s_r" % (name, tag)]
        _, _, core = check(cluster_emu, xyz, r, min_points)
        assert np.array_equal(core, z["%s_radius_%s_count" % (name, tag)] >= min_points)


@pytest.mark.parametrize("name", SCAN_NAMES)
@pytest.mark.parametrize("min_points", [1, 5, 15])
def test_reference_scans(cluster_emu, name, min_points):
    z = _golden("ref_scans.npz")
    xyz, r = z[name + "_xyz"], z[name + "_radius_r"]
    _, nc, core = check(cluster_emu, xyz, r, min_points)
    assert np.array_equal(core, z[name + "_radius_count"] >= min_points)
    assert nc >= 1


def test_line_at_exactly_r_and_one_float_closer(cluster_emu):
    # spacing r = 2^-4: every consecutive d2 == fl(r * r) exactly, so the line is one cluster
    r = F32(2.0 ** -4)
    x = np.arange(3000, dtype=np.float64) * float(r)
    xyz = np.stack([x, np.zeros_like(x), np.zeros_like(x)], 1).astype(F32)
    xyz = xyz[np.random.default_rng(1).permutation(len(xyz))]
    for mp in (1, 2, 3):
        labels, nc, core = check(cluster_emu, xyz, r, mp)
        assert nc == 1 and (labels == 0).all()
    labels, nc, core = check(cluster_emu, xyz, r, 4)
    assert nc == 0 and (labels == NOISE).all()
    # the radius one float below the spacing: the spacing is the next float above r, no pair is
    # within reach, so every point is noise for min_points >= 2 and its own cluster for 1
    rl = np.nextafter(r, F32(0))
    for mp in (2, 3):
        labels, nc, _ = check(cluster_emu, xyz, rl, mp)
        assert nc == 0 and (labels == NOISE).all()
    labels, nc, _ = check(cluster_emu, xyz, rl, 1)
    assert nc == len(xyz) and len(np.unique(labels)) == len(xyz)


@pytest.mark.parametrize("min_points", [0, 1, 2, 5, 10_000])
def test_duplicates(cluster_emu, min_points):
    rng = np.random.default_rng(2)
    base = rng.uniform(-1, 1, (300, 3)).astype(F32)
    xyz = np.concatenate([base, base[:100], base[:20], np.repeat(base[:1], 7, 0)])
    xyz = xyz[rng.permutation(len(xyz))]
    labels, nc, core = check(cluster_emu, xyz, 0.15, min_points)
    if min_points <= 1:
        assert core.all() and (labels != NOISE).all()
    if min_points > len(xyz):
        assert nc == 0 and (labels == NOISE).all()


def test_empty_index_and_voxel_grid(cluster_emu):
    labels, nc, core = cluster_emu.cluster(np.zeros((0, 3), F32), 0.1, 2)
    assert nc == 0 and len(labels) == 0
    rng = np.random.default_rng(3)
    xyz = rng.uniform(-1, 1, (4000, 3)).astype(F32)
    grid = ([-0.5, -0.6, -0.7], [0.5, 0.6, 0.4])
    for mp in (1, 4):
        labels, _, core = check(cluster_emu, xyz, 0.08, mp, voxel_grid=grid)
        outside = ~np.all((xyz >= F32(grid[0])) & (xyz <= F32(grid[1])), axis=1)
        assert outside.any() and (labels[outside] == NOISE).all() and not core[outside].any()
    # a voxel grid that holds no point: every point is noise
    labels, nc, _ = check(cluster_emu, xyz, 0.08, 1, voxel_grid=([5, 5, 5], [6, 6, 6]))
    assert nc == 0 and (labels == NOISE).all()


def test_blobs_and_offset_cloud(cluster_emu):
    rng = np.random.default_rng(4)
    centres = rng.uniform(-1, 1, (12, 3))
    blobs = centres[rng.integers(0, 12, 5000)] + 0.03 * rng.standard_normal((5000, 3))
    noise = rng.uniform(-1.1, 1.1, (250, 3))
    xyz = np.concatenate([blobs, noise]).astype(F32)
    for mp in (1, 4, 10):
        _, nc, _ = check(cluster_emu, xyz, 0.02, mp)
        assert nc >= 1
    far = (xyz + F32(1000.0)).astype(F32)
    for mp in (1, 6):
        check(cluster_emu, far, 0.02, mp)
