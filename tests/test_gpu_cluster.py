"""pcpx_cluster_by_density on the GPU against the brute-force DBSCAN of tests/emu_cluster_lib.py
(kd-tree candidates, the library's fp32 ball predicate, scipy's connected_components), label for
label; on the 10 M-point clouds against connected_components of the library's own radius_search
CSR and the density filter's mask.  The C++ call (tests/cpp/cluster_test.cpp) is compiled here
with strict warnings in the CPU suite and run on the GPU."""
import os
import subprocess
import threading

import numpy as np
import pytest

from emu_cluster_lib import NOISE, bruteforce_dbscan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz")
SCANS = os.path.join(ROOT, "tests", "golden", "ref_scans.npz")
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "cluster_test.cpp")
LIBDIR = os.path.join(ROOT, "point-cloud-processing_b200", "lib")
F32 = np.float32


def check(ix, xyz, r, min_points, indexed=None):
    """device labels == brute force; returns (labels, n_clusters)"""
    got, nc = ix.cluster_by_density(r, min_points)
    want, wnc, _ = bruteforce_dbscan(xyz, r, min_points, indexed)
    assert nc == wnc
    assert np.array_equal(got, want), np.nonzero(got != want)[0][:10]
    if min_points <= 1 and indexed is None:
        assert (got != NOISE).all()
    return got, nc


def compile_cpp(pcpx, exe):
    pcpx.lib()  # the library must exist to link against
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "include"), CPP_SRC, "-L", LIBDIR, "-lpcpx",
                    "-Wl,-rpath," + LIBDIR, "-o", str(exe)], check=True)


def test_cpp_cluster_compiles(pcpx, tmp_path):
    exe = tmp_path / "cluster_test"
    compile_cpp(pcpx, exe)
    if pcpx.device_count() == 0:
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU path" in r.stderr


@pytest.mark.gpu
def test_cpp_cluster_matches_brute_force(pcpx, tmp_path):
    exe = tmp_path / "cluster_test"
    compile_cpp(pcpx, exe)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks hold" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("name", CLOUDS + SCAN_NAMES)
def test_reference_clouds(pcpx, name):
    if name in CLOUDS:
        z = np.load(FIX)
        xyz, r = z[name + "_xyz"], F32(z[name + "_radius_0.02_r"])
    else:
        z = np.load(SCANS)
        xyz, r = z[name + "_xyz"], F32(z[name + "_radius_r"])
    with pcpx.Index(xyz) as ix:
        for rr in (r, F32(2) * r):
            for mp in (1, 5, 15):
                check(ix, xyz, rr, mp)


@pytest.mark.gpu
def test_gaussian_blobs_1m(pcpx):
    rng = np.random.default_rng(5)
    centres = rng.uniform(0, 10, (500, 3))
    blobs = centres[rng.integers(0, 500, 950_000)] + 0.04 * rng.standard_normal((950_000, 3))
    noise = rng.uniform(-0.2, 10.2, (50_000, 3))
    xyz = np.concatenate([blobs, noise]).astype(F32)
    xyz = xyz[rng.permutation(len(xyz))]
    with pcpx.Index(xyz) as ix:
        mbar = float(ix.radius_count(None, 0.02).mean())
        assert 10 < mbar < 60
        for mp in (1, 8):
            _, nc = check(ix, xyz, 0.02, mp)
            assert nc >= 500


@pytest.mark.gpu
def test_union_find_stress(pcpx):
    r = F32(0.01)
    # a straight chain of 1 M points 0.75 r apart: one cluster of diameter 10^6 edges
    n = 1_000_000
    x = np.arange(n, dtype=np.float64) * 0.75 * float(r)
    chain = np.stack([x, np.zeros(n), np.zeros(n)], 1).astype(F32)
    chain = chain[np.random.default_rng(6).permutation(n)]
    with pcpx.Index(chain) as ix:
        for mp in (1, 3):
            labels, nc = ix.cluster_by_density(r, mp)
            assert nc == 1 and (labels == 0).all()
        labels, nc = ix.cluster_by_density(r, 4)
        assert nc == 0 and (labels == NOISE).all()
    # a serpentine: rows 2 r apart joined at alternating ends, so the chain runs against the
    # Morton order of the cells and its smallest sorted position is far from most of it
    rows, per_row = 200, 1000
    pts = []
    for k in range(rows):
        xs = np.arange(per_row) * 0.75 * float(r)
        if k % 2:
            xs = xs[::-1]
        pts.append(np.stack([xs, np.full(per_row, 2.0 * k * float(r)), np.zeros(per_row)], 1))
        if k + 1 < rows:  # the link to the next row, at this row's end
            y = np.arange(1, 3) * 0.75 * float(r) * (2.0 / 2.25) + 2.0 * k * float(r)
            pts.append(np.stack([np.full(2, xs[-1]), y, np.zeros(2)], 1))
    snake = np.concatenate(pts).astype(F32)
    snake = snake[np.random.default_rng(7).permutation(len(snake))]
    with pcpx.Index(snake) as ix:
        labels, nc = check(ix, snake, r, 1)
        assert nc == 1
        check(ix, snake, r, 3)
    # 5 000 copies of one point: every ball holds the whole set
    dup = np.tile(np.array([[0.25, -1.5, 3.0]], F32), (5000, 1))
    with pcpx.Index(dup) as ix:
        for mp in (0, 1, 5000):
            labels, nc = ix.cluster_by_density(r, mp)
            assert nc == 1 and (labels == 0).all()
        labels, nc = ix.cluster_by_density(r, 5001)
        assert nc == 0 and (labels == NOISE).all()
    # a dense lattice: every point core, one cluster
    m = 64
    g = np.arange(m) * 0.5 * float(r)
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3).astype(F32)
    with pcpx.Index(lat) as ix:
        labels, nc = check(ix, lat, r, 10)  # a corner's ball holds 11 points
        assert nc == 1 and (labels == 0).all()


@pytest.mark.gpu
def test_border_ties_and_edge_cases(pcpx):
    xyz = np.array([[0, 0, 0], [0.5, 0, 0], [0, 0.5, 0], [0, 0, 0.5],
                    [3, 0, 0], [2.5, 0, 0], [3, 0.5, 0], [3, 0, 0.5],
                    [1.5, 5, 0], [1.5, 0, 0], [40, 40, 40]], F32)
    with pcpx.Index(xyz) as ix:
        labels, nc = check(ix, xyz, 1.0, 4)
        assert nc == 2 and labels.tolist() == [0, 0, 0, 0, 1, 1, 1, 1, NOISE, 0, NOISE]
    # blob B listed first: B is cluster 0 and the tie goes to B's point, now the lower index
    perm = [4, 5, 6, 7, 0, 1, 2, 3, 8, 9, 10]
    with pcpx.Index(xyz[perm]) as ix:
        labels, nc = check(ix, xyz[perm], 1.0, 4)
        assert labels.tolist() == [0, 0, 0, 0, 1, 1, 1, 1, NOISE, 0, NOISE]
        for r in (0.0, -1.0, np.inf):
            check(ix, xyz[perm], r, 2)
        with pytest.raises(pcpx.PcpxError):
            ix.cluster_by_density(np.nan, 2)
        assert pcpx.lib().pcpx_cluster_by_density(ix._h, 1.0, 2, None, None) != 0
    with pcpx.Index(np.zeros((0, 3), F32)) as ix:
        labels, nc = ix.cluster_by_density(0.1, 2)
        assert nc == 0 and len(labels) == 0
    # a voxel grid: the points it leaves out are noise, and count in no ball
    cube = pcpx.synth.uniform_cube(100_000, half=1.0)
    grid = ([-0.5, -0.6, -0.7], [0.5, 0.6, 0.4])
    indexed = np.all((cube >= F32(grid[0])) & (cube <= F32(grid[1])), axis=1)
    with pcpx.Index(cube, voxel_grid=grid) as ix:
        for mp in (1, 6):
            labels, _ = check(ix, cube, 0.05, mp, indexed=indexed)
            assert (labels[~indexed] == NOISE).all()
    far = (cube + F32(1000.0)).astype(F32)
    with pcpx.Index(far) as ix:
        check(ix, far, 0.05, 6)


def _csr_dbscan(xyz, off, idx, core):
    """labels of the contract from the library's own radius_search CSR and a core mask"""
    from scipy.sparse import csr_matrix
    from scipy.sparse.csgraph import connected_components

    n = len(xyz)
    rows = np.repeat(np.arange(n, dtype=np.int32), np.diff(off).astype(np.int64))
    cols = idx.view(np.int32)
    keep = core[rows] & core[cols]
    g = csr_matrix((np.ones(int(keep.sum()), np.int8), (rows[keep], cols[keep])), shape=(n, n))
    _, comp = connected_components(g, directed=False)
    labels = np.full(n, NOISE, np.uint32)
    # components are numbered by their smallest vertex; the core ones keep that order
    _, labels[core] = np.unique(comp[core], return_inverse=True)
    b = ~core[rows] & core[cols]
    bi, bj = rows[b], cols[b]
    d = xyz[bi] - xyz[bj]
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    order = np.lexsort((bj, d2, bi))
    bi, bj = bi[order], bj[order]
    firsts = np.ones(len(bi), bool)
    firsts[1:] = bi[1:] != bi[:-1]
    labels[bi[firsts]] = labels[bj[firsts]]
    return labels, int(core.any() and labels[core].max() + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("cloud", ["plane", "mix"])
def test_10m_against_radius_search_csr(pcpx, cloud):
    n = 10_000_000
    xyz = pcpx.synth.noisy_plane(n) if cloud == "plane" else pcpx.synth.noise_mix(n)
    with pcpx.Index(xyz) as ix:
        r = 0.01 if cloud == "plane" else float(ix.mean_knn_distance(15)[1])
        labels, nc = ix.cluster_by_density(r, 5)
        mask, _, _ = ix.density_filter(r, 5, want_points=False)
        off, idx = ix.radius_search(None, r)
    core = mask.astype(bool)
    assert (labels[core] != NOISE).all()
    want, wnc = _csr_dbscan(xyz, off, idx, core)
    del off, idx
    assert nc == wnc
    assert np.array_equal(labels, want)
    if cloud == "plane":
        assert nc < 100 and np.bincount(labels[labels != NOISE]).max() > 0.95 * n


@pytest.mark.gpu
def test_identical_bytes_across_buffers_handles_and_threads(pcpx):
    import torch

    xyz = pcpx.synth.noise_mix(300_000, seed=3)
    r = 0.02
    L = pcpx.lib()
    with pcpx.Index(xyz) as ix:
        h_labels, h_nc = ix.cluster_by_density(r, 5)
        assert h_nc > 1 and (h_labels == NOISE).any()
        d = torch.empty(len(xyz), dtype=torch.int32, device="cuda")
        d_labels, d_nc = ix.cluster_by_density(r, 5, out_labels=d)
        assert d_nc == h_nc
        assert np.array_equal(d_labels.cpu().numpy().view(np.uint32), h_labels)
        assert ix.timings()["kernel_launches"] == 8
        assert L.pcpx_cluster_by_density(ix._h, r, 5, h_labels.ctypes.data, None) == 0
        want = [ix.cluster_by_density(r * (1 + 0.5 * i), 2 + i) for i in range(4)]
        got, errors = [None] * 4, []

        def run(i):
            try:
                got[i] = ix.cluster_by_density(r * (1 + 0.5 * i), 2 + i)
            except Exception as e:  # surfaced below
                errors.append(e)

        threads = [threading.Thread(target=run, args=(i,)) for i in range(4)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors
        for g, w in zip(got, want):
            assert g[1] == w[1] and np.array_equal(g[0], w[0])
    os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"] = "1"
    try:
        with pcpx.Index(xyz, devices=[0, 0]) as many:
            m_labels, m_nc = many.cluster_by_density(r, 5)
            assert m_nc == h_nc and np.array_equal(m_labels, h_labels)
    finally:
        del os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"]
