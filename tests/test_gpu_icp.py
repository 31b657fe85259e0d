"""pcpx_nearest_within and pcpx_icp on the GPU: the bounded nearest neighbour against the kd-tree
brute force of tests/emu_icp_lib.py (index for index, d2 bit for bit) and against knn(k = 1); one
ICP step against a numpy step (brute-force pairs, fp64 sums, eigh / SVD solve); recovery of known
rigid motions on the reference scans and synthetic clouds; identical bytes across buffers,
strides, threads and replicas; the edge cases.  The C++ call (tests/cpp/icp_test.cpp) is compiled
with strict warnings in the CPU suite and run here."""
import os
import subprocess
import threading

import numpy as np
import pytest

from emu_icp_lib import (NONE, brute_nearest_within, np_step, pose_error, rigid,
                         transform_f32)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz")
SCANS = os.path.join(ROOT, "tests", "golden", "ref_scans.npz")
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "icp_test.cpp")
LIBDIR = os.path.join(ROOT, "point-cloud-processing_b200", "lib")
F32 = np.float32


def _cloud(name):
    if name in CLOUDS:
        return np.load(FIX)[name + "_xyz"].astype(F32)
    return np.load(SCANS)[name + "_xyz"].astype(F32)


def _extent(xyz):
    return float(np.linalg.norm(xyz.max(0).astype(np.float64) - xyz.min(0)))


def _centre(ix):
    lo, hi = ix.bbox()
    return 0.5 * (lo.astype(np.float64) + hi.astype(np.float64))


def check_nearest(pcpx, xyz, q, r, T=None, voxel_grid=None, ix=None):
    indexed = None
    if voxel_grid is not None:
        lo, hi = (np.asarray(v, F32) for v in voxel_grid)
        indexed = np.all((xyz >= lo) & (xyz <= hi), axis=1)
    own = ix is None
    ix = pcpx.Index(xyz, voxel_grid=voxel_grid) if own else ix
    try:
        got_i, got_d = ix.nearest_within(q, r, T)
    finally:
        if own:
            ix.close()
    y = q if T is None else transform_f32(q, T)
    want_i, want_d = brute_nearest_within(xyz, y, r, indexed)
    assert np.array_equal(got_i, want_i), np.nonzero(got_i != want_i)[0][:10]
    assert np.array_equal(got_d.view(np.uint32), want_d.view(np.uint32))
    return got_i, got_d


def compile_cpp(pcpx, exe):
    pcpx.lib()  # the library must exist to link against
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "include"), CPP_SRC, "-L", LIBDIR, "-lpcpx",
                    "-Wl,-rpath," + LIBDIR, "-o", str(exe)], check=True)


def test_cpp_icp_compiles(pcpx, tmp_path):
    exe = tmp_path / "icp_test"
    compile_cpp(pcpx, exe)
    if pcpx.device_count() == 0:
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU path" in r.stderr


@pytest.mark.gpu
def test_cpp_icp_registers(pcpx, tmp_path):
    exe = tmp_path / "icp_test"
    compile_cpp(pcpx, exe)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks hold" in r.stdout


# ---- nearest_within ------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("name", CLOUDS + SCAN_NAMES)
def test_nearest_within_reference_clouds(pcpx, name):
    xyz = _cloud(name)
    ext = _extent(xyz)
    rng = np.random.default_rng(1)
    q = xyz[rng.integers(0, len(xyz), 20000)] + rng.normal(0, 0.01 * ext, (20000, 3)).astype(F32)
    T = rigid(4.0, [1, 2, 3], 0.01 * ext * np.array([1, -1, 0.5]))
    with pcpx.Index(xyz) as ix:
        for r in (0.005 * ext, 0.03 * ext, 2.0 * ext):
            check_nearest(pcpx, xyz, q, r, ix=ix)
            check_nearest(pcpx, xyz, q, r, T, ix=ix)
        _, d2 = check_nearest(pcpx, xyz, xyz, 0.01 * ext, ix=ix)
        assert (d2 == 0).all()


@pytest.mark.gpu
def test_nearest_within_geometry_cases(pcpx):
    g = np.arange(8, dtype=F32)
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    q = np.concatenate([lat[:200] + F32(0.5), lat[:200] + np.array([0.5, 0.5, 0], F32),
                        lat[:200] + np.array([0.5, 0, 0], F32)])
    for r in (0.5, 0.8660254, 3.0):
        check_nearest(pcpx, lat, q, r)
    r = F32(0.25)
    line = np.zeros((64, 3), F32)
    line[:, 0] = np.arange(64, dtype=F32) * r
    got, _ = check_nearest(pcpx, line[::2], line[1::2], r)
    assert (got[:-1] != NONE).all()
    got, _ = check_nearest(pcpx, line[::2], line[1::2], np.nextafter(r, F32(0)))
    assert (got == NONE).all()
    rng = np.random.default_rng(3)
    xyz = rng.uniform(0, 1, (50000, 3)).astype(F32)
    far = rng.uniform(-1, 2, (20000, 3)).astype(F32)
    check_nearest(pcpx, xyz, far, 0.05)
    check_nearest(pcpx, xyz, far, 0.6)
    bad = far[:60].copy()
    bad[::3, 0] = np.nan
    bad[1::3, 2] = -np.inf
    got, d2 = check_nearest(pcpx, xyz, bad, 10.0)
    assert (got[::3] == NONE).all() and (got[1::3] == NONE).all()
    vox = (np.array([0.2, 0.2, 0.2], F32), np.array([0.7, 0.8, 0.9], F32))
    check_nearest(pcpx, xyz, far, 0.1, voxel_grid=vox)
    off = xyz + F32(1000)
    check_nearest(pcpx, off, far + F32(1000), 0.05)
    check_nearest(pcpx, off, off, 0.02, rigid(3, [0, 0, 1], [0.01, 0, 0]))


@pytest.mark.gpu
def test_nearest_within_scan_1m(pcpx):
    xyz = pcpx.synth.scan(1_000_000)
    ext = _extent(xyz)
    rng = np.random.default_rng(2)
    lo, hi = xyz.min(0), xyz.max(0)
    q = rng.uniform(lo - 0.05 * (hi - lo), hi + 0.05 * (hi - lo), (1_000_000, 3)).astype(F32)
    q[: len(q) // 2] = xyz[rng.integers(0, len(xyz), len(q) // 2)] + \
        rng.normal(0, 0.002 * ext, (len(q) // 2, 3)).astype(F32)
    with pcpx.Index(xyz) as ix:
        check_nearest(pcpx, xyz, q, 0.01 * ext, ix=ix)
        t = ix.timings()
        assert t["kernel_launches"] >= 2


@pytest.mark.gpu
def test_nearest_within_equals_knn_noise_mix_10m(pcpx):
    xyz = pcpx.synth.noise_mix(10_000_000)
    q = pcpx.synth.noise_mix(10_000_000, seed=12)
    with pcpx.Index(xyz) as ix:
        ki, kd, _ = ix.knn(q, 1, eps=0.0)
        ki, kd = ki[:, 0], kd[:, 0]
        spacing = float(np.sqrt(np.median(kd)))
        for r in (spacing, 4 * spacing):
            gi, gd = ix.nearest_within(q, r)
            inside = kd <= F32(r) * F32(r)
            assert inside.any() and (~inside).any()
            assert np.array_equal(gi[inside], ki[inside])
            assert np.array_equal(gd[inside].view(np.uint32), kd[inside].view(np.uint32))
            assert (gi[~inside] == NONE).all() and np.isinf(gd[~inside]).all()


# ---- ICP -----------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("metric", ["point_to_plane", "point_to_point"])
@pytest.mark.parametrize("name", ["stanford_bunny", "fandisk"])
def test_one_step_equals_numpy(pcpx, name, metric):
    m = 0 if metric == "point_to_plane" else 1
    xyz = _cloud(name)
    ext = _extent(xyz)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        c = _centre(ix)
        src = transform_f32(xyz, rigid(5, [1, 1, 0], 0.01 * ext * np.ones(3)))
        for init in (np.eye(4), rigid(-3, [0, 0, 1], [0.005 * ext, 0, 0]),
                     rigid(8, [1, -2, 0.5], -0.01 * ext * np.ones(3))):
            corr = np.zeros(len(src), np.uint32)
            T, res = ix.icp(src, 0.05 * ext, nrm, metric, init=init, max_iterations=1,
                            out_correspondences=corr)
            W, s = np_step(m, xyz, nrm, src, 0.05 * ext, init, c)
            assert res["iterations"] == 1
            assert np.abs(T[:3, :3] - W[:3, :3]).max() < 1e-9
            assert np.abs(T[:3, 3] - W[:3, 3]).max() < 1e-9 * ext
            want, _ = brute_nearest_within(xyz, transform_f32(src, T), 0.05 * ext)
            assert np.array_equal(corr, want)
            assert res["n_correspondences"] == int((want != NONE).sum())


def _recover(pcpx, xyz, metric, angle, axis, frac, max_distance_frac=0.05, tol=1e-5):
    ext = _extent(xyz)
    M = rigid(angle, axis, frac * ext * np.array(axis) / np.linalg.norm(axis))
    src = transform_f32(xyz, M)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(src, max_distance_frac * ext, nrm, metric, max_iterations=100)
    ang, dist = pose_error(T, np.linalg.inv(M))
    assert res["stop_reason"] == "converged", res
    assert ang < tol and dist < tol * ext, (ang, dist / ext, res)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCAN_NAMES)
def test_recovery_on_scans(pcpx, name):
    # point-to-plane: point-to-point steps shrink below the tolerances while still off the
    # answer on these scans (fandisk, 2 degrees: stopped 5e-3 rad away), as point-to-point ICP does
    _recover(pcpx, _cloud(name), "point_to_plane", 6, [1, -2, 1], 0.015)
    _recover(pcpx, _cloud(name), "point_to_plane", 2, [0, 1, 0.3], 0.005)


@pytest.mark.gpu
def test_recovery_scan_1m(pcpx):
    xyz = pcpx.synth.scan(1_000_000)
    res = _recover(pcpx, xyz, "point_to_plane", 10, [1, 1, 2], 0.02)
    assert res["fitness"] > 0.95


@pytest.mark.gpu
def test_recovery_separate_noisy_sample(pcpx):
    # a second noisy sample of the bunny's surface: its points jittered by 0.1 % of the extent;
    # the motion is recovered to 2e-3 rad and 2e-3 x the extent
    xyz = _cloud("stanford_bunny")
    ext = _extent(xyz)
    rng = np.random.default_rng(8)
    other = (xyz + rng.normal(0, 1e-3 * ext, xyz.shape)).astype(F32)
    M = rigid(5, [1, 0, 1], 0.01 * ext * np.array([1, 0, -1]))
    src = transform_f32(other, M)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(src, 0.05 * ext, nrm, max_iterations=100)
    ang, dist = pose_error(T, np.linalg.inv(M))
    assert ang < 2e-3 and dist < 2e-3 * ext, (ang, dist / ext, res)


@pytest.mark.gpu
def test_recovery_partial_overlap(pcpx):
    # the source is half of the target (a box crop), moved: 50 % overlap
    xyz = _cloud("stanford_bunny")
    ext = _extent(xyz)
    crop = xyz[xyz[:, 0] < np.median(xyz[:, 0])]
    M = rigid(4, [0, 1, 1], 0.01 * ext * np.array([0, 1, 1]))
    src = transform_f32(crop, M)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(src, 0.03 * ext, nrm, max_iterations=100)
    ang, dist = pose_error(T, np.linalg.inv(M))
    assert res["stop_reason"] == "converged"
    assert ang < 1e-5 and dist < 1e-5 * ext, (ang, dist / ext, res)


@pytest.mark.gpu
def test_degenerate_plane(pcpx):
    # plane to plane: the offset along the normal and the tilt are recovered; the motions the
    # pairs do not constrain (in-plane sliding, spin about the normal) stay (nearly) zero
    xyz = pcpx.synth.noisy_plane(200_000)
    ext = _extent(xyz)
    M = rigid(1.0, [1, 0, 0], [0, 0, 0.01 * ext])
    src = transform_f32(xyz, M)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(src, 0.05 * ext, nrm, max_iterations=50)
    y = transform_f32(src, T)
    # the moved plane is back on z = 0 (to the noise) and level
    assert abs(float(np.mean(y[:, 2].astype(np.float64) - xyz[:, 2]))) < 1e-4 * ext
    A = np.c_[y[:, :2].astype(np.float64), np.ones(len(y))]
    slope = np.linalg.lstsq(A, y[:, 2].astype(np.float64), rcond=None)[0][:2]
    assert np.abs(slope).max() < 1e-4
    # in-plane motion of T about the centre: small against the extent
    D = T @ M
    assert np.abs(D[:2, 3]).max() < 1e-2 * ext
    assert abs(np.arctan2(D[1, 0], D[0, 0])) < 1e-2


@pytest.mark.gpu
def test_identical_bytes(pcpx):
    import torch

    xyz = _cloud("spray")
    ext = _extent(xyz)
    src = transform_f32(xyz[::2], rigid(5, [1, 2, 0], 0.01 * ext * np.ones(3)))
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        args = dict(max_distance=0.05 * ext, max_iterations=40)

        def run(source, normals=nrm, stride=12, target=ix):
            corr = np.zeros(len(src), np.uint32)
            T, res = target.icp(source, normals=normals, out_correspondences=corr,
                                source_stride_bytes=stride, **args)
            return T.tobytes(), tuple(res.values()), corr.tobytes()

        ref = run(src)
        assert run(src) == ref
        dev = torch.from_numpy(src).cuda()
        assert run(dev, torch.from_numpy(nrm).cuda()) == ref
        padded = np.zeros((len(src), 5), F32)
        padded[:, :3] = src
        assert run(padded, stride=20) == ref
        out = [None] * 4

        def worker(i):
            out[i] = run(src)

        threads = [threading.Thread(target=worker, args=(i,)) for i in range(4)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert all(o == ref for o in out)
    os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"] = "1"
    try:
        with pcpx.Index(xyz, devices=[0, 0]) as many:
            assert run(src, target=many) == ref
    finally:
        del os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"]


@pytest.mark.gpu
def test_edge_cases(pcpx):
    xyz = _cloud("fandisk")
    ext = _extent(xyz)
    init = rigid(3, [0, 0, 1], [1, 2, 3])
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(np.zeros((0, 3), F32), 1.0, nrm, init=init)
        assert np.array_equal(T, init) and res["n_correspondences"] == 0 and np.isnan(res["rmse"])
        for bad in (np.nan, np.inf, 0.0, -1.0):
            with pytest.raises(pcpx.PcpxError) as e:
                ix.icp(xyz, bad, nrm)
            assert e.value.code == -1
            with pytest.raises(pcpx.PcpxError):
                ix.nearest_within(xyz, bad)
        with pytest.raises(pcpx.PcpxError):
            ix.icp(xyz, 1.0, nrm, metric=7)
        with pytest.raises(pcpx.PcpxError):
            ix.icp(xyz, 1.0, None, metric="point_to_plane")
        # the ways to stop
        _, res = ix.icp(xyz, 0.05 * ext, nrm, max_iterations=100)
        assert res["stop_reason"] == "converged" and res["fitness"] == 1.0 and res["rmse"] == 0
        moved = transform_f32(xyz, rigid(5, [1, 0, 0], [0.01 * ext, 0, 0]))
        _, res = ix.icp(moved, 0.05 * ext, nrm, max_iterations=2, rotation_tolerance=1e-300,
                        translation_tolerance=1e-300)
        assert res["stop_reason"] == "max_iterations" and res["iterations"] == 2
        far = xyz + F32(10 * ext)
        corr = np.zeros(len(far), np.uint32)
        T, res = ix.icp(far, 0.05 * ext, nrm, out_correspondences=corr)
        assert res["stop_reason"] == "too_few" and res["iterations"] == 0
        assert np.array_equal(T, np.eye(4)) and (corr == NONE).all()
        nan_n = nrm.copy()
        nan_n[:] = np.nan
        _, res = ix.icp(xyz, 0.05 * ext, nan_n)
        assert res["stop_reason"] == "too_few" and res["n_correspondences"] == 0
        _, res = ix.icp(xyz, 0.05 * ext, nan_n, metric="point_to_point")
        assert res["stop_reason"] == "converged"
        t = ix.timings()
        assert t["kernel_launches"] >= 4 and t["total_ms"] > 0
    with pcpx.Index(np.zeros((0, 3), F32)) as empty:
        corr = np.zeros(len(xyz), np.uint32)
        T, res = empty.icp(xyz, 1.0, metric="point_to_point", init=init, out_correspondences=corr)
        assert np.array_equal(T, init) and res["n_correspondences"] == 0
        assert (corr == NONE).all()
        gi, gd = empty.nearest_within(xyz, 1.0)
        assert (gi == NONE).all() and np.isinf(gd).all()


@pytest.mark.gpu
def test_scan_10m_converges(pcpx):
    xyz = pcpx.synth.scan(10_000_000)
    ext = _extent(xyz)
    M = rigid(3, [1, 2, 3], 0.005 * ext * np.array([1, -1, 0]))
    src = transform_f32(xyz, M)
    with pcpx.Index(xyz) as ix:
        nrm = ix.estimate_normals(None, 15)
        T, res = ix.icp(src, 0.02 * ext, nrm, max_iterations=100)
    ang, dist = pose_error(T, np.linalg.inv(M))
    assert res["stop_reason"] == "converged", res
    assert ang < 1e-5 and dist < 1e-5 * ext, (ang, dist / ext)
