"""pcpx_estimate_normals_radius / pcpx_estimate_tangent_planes_radius on the GPU against the
CPU checker (tests/ball_oracle.py).  Counts bit-exact against radius_count; normals
1 - |cos| <= 1e-4 where the eigengap > 1e-3; centroids within 1e-5 * max(1, max|p|) of the
fp64 mean of the exact ball.  The C++ drop-in (pcp::gpu_radius_map) is compiled here with
strict warnings in the CPU suite and run on the GPU."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

from ball_oracle import (bruteforce_ball_normals, centroid_tolerance, normal_error,
                         radius_normals)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz")
SCANS = os.path.join(ROOT, "tests", "golden", "ref_scans.npz")
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "radius_normals_test.cpp")
LIBDIR = os.path.join(ROOT, "point-cloud-processing_b200", "lib")
UP = np.float32([0, 0, 1])


def check(xyz, got, want):
    """got = (normals, centroids, counts); want = (normals, centroids, gaps, counts)"""
    nrm, ctr, cnt = got
    wnrm, wctr, gap, wcnt = want
    assert np.array_equal(np.asarray(cnt, np.uint32), wcnt)
    well = gap > 1e-3
    if well.any():
        assert normal_error(nrm, wnrm)[well].max() <= 1e-4
    full = wcnt > 0
    assert np.isnan(ctr[~full]).all() and (nrm[~full] == UP).all()
    if full.any():
        assert np.abs(ctr[full] - wctr[full]).max() <= centroid_tolerance(xyz)
    assert np.allclose(np.linalg.norm(nrm, axis=1), 1, atol=1e-5)


def radius_for(xyz, m):
    """a radius whose ball holds about m points on average (from the mean 8-NN distance)"""
    from scipy.spatial import cKDTree

    d, _ = cKDTree(xyz).query(xyz[:: max(1, len(xyz) // 2000)], 9)
    return float(np.float32(np.median(d[:, 8]) * np.sqrt(m / 9.0)))


def compile_cpp(pcpx, exe):
    pcpx.lib()  # the library must exist to link against
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "include"), CPP_SRC, "-L", LIBDIR, "-lpcpx",
                    "-Wl,-rpath," + LIBDIR, "-o", str(exe)], check=True)


def test_dropin_radius_map_compiles(pcpx, tmp_path):
    exe = tmp_path / "radius_normals_test"
    compile_cpp(pcpx, exe)
    if pcpx.device_count() == 0:
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU path" in r.stderr  # fails loudly without a GPU


@pytest.mark.gpu
def test_dropin_radius_map_matches_lambdas(pcpx, tmp_path):
    exe = tmp_path / "radius_normals_test"
    compile_cpp(pcpx, exe)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks hold" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("name", CLOUDS)
def test_reference_fixture_clouds(pcpx, oracle, name):
    fix = np.load(FIX)
    xyz, q = fix[name + "_xyz"], fix[name + "_queries"]
    oc = oracle.cloud(xyz)
    with pcpx.Index(xyz) as ix:
        for m in (8, 32, 200):
            r = radius_for(xyz, m)
            for queries in (None, q):
                pts, nrm, cnt = ix.estimate_tangent_planes_radius(queries, r)
                # r > 1 (the cube): the exact ball, which the reference's own prune can miss
                check(xyz, (nrm, pts, cnt), radius_normals(oc, queries, r, exact_prune=int(r > 1)))
                assert np.array_equal(cnt, ix.radius_count(queries, r))
                assert np.array_equal(ix.estimate_normals_radius(queries, r), nrm)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCAN_NAMES)
def test_reference_scans(pcpx, oracle, name):
    scans = np.load(SCANS)
    xyz, r = scans[name + "_xyz"], float(scans[name + "_radius_r"])
    oc = oracle.cloud(xyz)
    with pcpx.Index(xyz) as ix:
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(None, r)
        assert np.array_equal(cnt, scans[name + "_radius_count"])
        check(xyz, (nrm, pts, cnt), radius_normals(oc, None, r))
        q = (xyz[::7] + np.float32(0.3 * r)).astype(np.float32)
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(q, r)
        check(xyz, (nrm, pts, cnt), radius_normals(oc, q, r))


@pytest.mark.gpu
def test_composition_gives_the_same_normals(pcpx, oracle):
    xyz = pcpx.synth.noisy_sphere(20_000, seed=5)
    r = radius_for(xyz, 32)
    oc = oracle.cloud(xyz)
    with pcpx.Index(xyz) as ix:
        off, idx = ix.radius_search(None, r)
        composed = pcpx.normals_from_neighbourhoods(xyz[idx.astype(np.int64)], off)
        cnt = np.zeros(len(xyz), np.uint32)
        fused = ix.estimate_normals_radius(None, r, out_count=cnt)
        assert np.array_equal(cnt, ix.radius_count(None, r))
        assert np.array_equal(cnt, np.diff(off.astype(np.int64)))
        gap = radius_normals(oc, None, r)[2]
        well = gap > 1e-3
        assert well.mean() > 0.99
        assert normal_error(fused, composed)[well].max() <= 1e-4


@pytest.mark.gpu
def test_edge_cases(pcpx):
    xyz = pcpx.synth.noisy_plane(5000, extent=1.0)
    with pcpx.Index(xyz) as ix:
        # nq = 0
        out = ix.estimate_normals_radius(np.zeros((0, 3), np.float32), 0.05)
        assert out.shape == (0, 3)
        assert pcpx.lib().pcpx_estimate_normals_radius(ix._h, None, 0, 12, None, 0.05, None,
                                                        None) == 0
        # a NULL required output
        q = np.ascontiguousarray(xyz[:4])
        assert pcpx.lib().pcpx_estimate_normals_radius(ix._h, q.ctypes.data, 4, 12, None, 0.05,
                                                        None, None) == -1
        nrm = np.zeros((4, 3), np.float32)
        assert pcpx.lib().pcpx_estimate_tangent_planes_radius(
            ix._h, q.ctypes.data, 4, 12, None, 0.05, None, nrm.ctypes.data, None) == -1
        # a far external query: (0,0,1), NaN centroid, count 0
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(np.float32([[50, 50, 50]]), 0.05)
        assert cnt[0] == 0 and np.isnan(pts).all() and (nrm == UP).all()
        # r = 0: every point alone in its ball (the cloud has no duplicates)
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(None, 0.0)
        assert (cnt == 1).all() and (nrm == UP).all() and np.array_equal(pts, xyz)
    # balls of one and two points
    two = np.float32([[0, 0, 0], [0.01, 0, 0], [5, 5, 5]])
    with pcpx.Index(two) as ix:
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(None, 0.02)
        assert list(cnt) == [2, 2, 1]
        assert np.allclose(pts[:2], [[0.005, 0, 0]] * 2) and np.array_equal(pts[2], two[2])
        assert (nrm[2] == UP).all()
        assert np.abs(nrm[:2, 0]).max() < 1e-6  # any direction across the segment
        assert np.allclose(np.linalg.norm(nrm, axis=1), 1, atol=1e-6)


@pytest.mark.gpu
def test_radius_above_one_is_the_exact_ball(pcpx):
    rng = np.random.default_rng(8)
    xyz = rng.uniform(-3, 3, (3000, 3)).astype(np.float32)
    xyz[:, 2] *= np.float32(0.1)
    q = rng.uniform(-3, 3, (150, 3)).astype(np.float32)
    with pcpx.Index(xyz) as ix:
        for r in (1.5, 2.5):
            pts, nrm, cnt = ix.estimate_tangent_planes_radius(q, r)
            check(xyz, (nrm, pts, cnt), bruteforce_ball_normals(xyz, q, r))


@pytest.mark.gpu
def test_voxel_grid_unindexed_points_are_queries_only(pcpx, oracle):
    rng = np.random.default_rng(6)
    xyz = rng.uniform(-2, 2, (8000, 3)).astype(np.float32)
    xyz[:, 2] *= np.float32(0.05)
    box = (np.float32([-1, -1, -1]), np.float32([1, 1, 1]))
    oc = oracle.cloud(xyz, bbox=np.concatenate(box))
    with pcpx.Index(xyz, voxel_grid=box) as ix:
        assert ix.info()["n_indexed"] < len(xyz)
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(None, 0.15)
        check(xyz, (nrm, pts, cnt), radius_normals(oc, None, 0.15))
        inside = (np.abs(xyz) <= 1).all(1)
        check(xyz, (nrm, pts, cnt), bruteforce_ball_normals(xyz[inside], xyz, 0.15))


@pytest.mark.gpu
def test_identical_bytes_across_buffers_and_handles(pcpx):
    import torch

    xyz = pcpx.synth.noise_mix(200_000, seed=3)
    rng = np.random.default_rng(4)
    q = (xyz[rng.choice(len(xyz), 20_000, replace=False)]
         + rng.normal(0, 1e-3, (20_000, 3))).astype(np.float32)
    radii = rng.uniform(0, 0.03, len(q)).astype(np.float32)
    r = 0.01
    with pcpx.Index(xyz) as ix:
        h_pts, h_nrm, h_cnt = ix.estimate_tangent_planes_radius(q, r, radii=radii)
        # device queries, radii and outputs
        d_pts, d_nrm, d_cnt = ix.estimate_tangent_planes_radius(
            torch.from_numpy(q).cuda(), r, radii=torch.from_numpy(radii).cuda())
        assert np.array_equal(d_nrm.cpu().numpy(), h_nrm)
        assert np.array_equal(d_pts.cpu().numpy(), h_pts, equal_nan=True)
        assert np.array_equal(d_cnt.cpu().numpy().astype(np.uint32), h_cnt)
        d_out = torch.empty((len(q), 3), dtype=torch.float32, device="cuda")
        d_c = torch.empty(len(q), dtype=torch.int32, device="cuda")
        ix.estimate_normals_radius(torch.from_numpy(q).cuda(), r, radii=torch.from_numpy(radii).cuda(),
                                   out=d_out, out_count=d_c)
        assert np.array_equal(d_out.cpu().numpy(), h_nrm)
        # strided queries (16-byte rows) from the host and from the device
        q4 = np.zeros((len(q), 4), np.float32)
        q4[:, :3] = q
        for src in (q4, torch.from_numpy(q4).cuda()):
            ptr = src.ctypes.data if isinstance(src, np.ndarray) else src.data_ptr()
            s_nrm = np.zeros((len(q), 3), np.float32)
            s_cnt = np.zeros(len(q), np.uint32)
            assert pcpx.lib().pcpx_estimate_normals_radius(
                ix._h, ptr, len(q), 16, radii.ctypes.data, C.c_float(r), s_nrm.ctypes.data,
                s_cnt.ctypes.data) == 0
            assert np.array_equal(s_nrm, h_nrm) and np.array_equal(s_cnt, h_cnt)
        self_one = ix.estimate_tangent_planes_radius(None, r)
    os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"] = "1"
    try:
        with pcpx.Index(xyz, devices=[0, 0]) as many:
            m_pts, m_nrm, m_cnt = many.estimate_tangent_planes_radius(q, r, radii=radii)
            assert np.array_equal(m_nrm, h_nrm) and np.array_equal(m_cnt, h_cnt)
            assert np.array_equal(m_pts, h_pts, equal_nan=True)
            for a, b in zip(many.estimate_tangent_planes_radius(None, r), self_one):
                assert np.array_equal(a, b, equal_nan=True)
    finally:
        del os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"]


@pytest.mark.gpu
def test_concurrent_calls_from_host_threads(pcpx):
    xyz = pcpx.synth.noisy_plane(300_000, extent=2.0)
    radii = [0.004, 0.006, 0.008, 0.01]
    with pcpx.Index(xyz) as ix:
        want = [ix.estimate_tangent_planes_radius(None, r) for r in radii]
        got = [None] * (2 * len(radii))
        errors = []

        def run(i):
            try:
                got[i] = ix.estimate_tangent_planes_radius(None, radii[i % len(radii)])
            except Exception as e:  # surfaced below
                errors.append(e)

        threads = [threading.Thread(target=run, args=(i,)) for i in range(len(got))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors
        for i, g in enumerate(got):
            for a, b in zip(g, want[i % len(radii)]):
                assert np.array_equal(a, b, equal_nan=True)


@pytest.mark.gpu
def test_offset_cloud_cancellation(pcpx, oracle):
    xyz = (pcpx.synth.noisy_plane(50_000, extent=1.0).astype(np.float64) + 1000.0).astype(np.float32)
    r = 0.02
    with pcpx.Index(xyz) as ix:
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(xyz[:3000], r)
    want = bruteforce_ball_normals(xyz, xyz[:3000], r)
    check(xyz, (nrm, pts, cnt), want)
    assert (want[2] > 1e-3).mean() > 0.95
    check(xyz, (nrm, pts, cnt), radius_normals(oracle.cloud(xyz), xyz[:3000], r))


@pytest.mark.gpu
def test_one_ball_of_thousands(pcpx):
    xyz = pcpx.synth.noisy_plane(100_000, extent=1.0)
    q = np.float32([[0.5, 0.5, 0.0], [0.2, 0.7, 0.0]])
    with pcpx.Index(xyz) as ix:
        pts, nrm, cnt = ix.estimate_tangent_planes_radius(q, 0.09)
    assert cnt.min() >= 2000
    check(xyz, (nrm, pts, cnt), bruteforce_ball_normals(xyz, q, 0.09))


@pytest.mark.gpu
def test_10m_plane(pcpx, oracle):
    xyz = pcpx.synth.noisy_plane(10_000_000)
    r = 0.01
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals_radius(None, r)
        cnt = np.zeros(len(xyz), np.uint32)
        pts, nrm2, cnt2 = ix.estimate_tangent_planes_radius(None, r)
        assert np.array_equal(nrm, nrm2)
        assert np.allclose(np.linalg.norm(nrm, axis=1), 1.0, atol=1e-5)
        assert np.array_equal(cnt2, ix.radius_count(None, r, out_count=cnt))
        assert 25 < cnt2.mean() < 40
        assert np.median(np.abs(nrm[:, 2])) > 0.95
    sample = np.sort(np.random.default_rng(12).choice(len(xyz), 10_000, replace=False))
    want = radius_normals(oracle.cloud(xyz), xyz[sample], r)
    check(xyz, (nrm[sample], pts[sample], cnt2[sample]), want)
    assert (want[2] > 1e-3).mean() > 0.99
