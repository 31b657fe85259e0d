"""pcpx_box_count / pcpx_box_search on the GPU against a numpy brute force of the fp32 predicate
min <= p <= max (tests/emu_box_lib.py: bruteforce_boxes).  Comparisons only: every checked box's
list is set-exact.  The C++ drop-in overloads (tests/cpp/box_search_test.cpp) are compiled here
with strict warnings in the CPU suite and run on the GPU."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

from emu_box_lib import bruteforce_boxes, split_csr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIX = os.path.join(ROOT, "tests", "golden", "ref_fixtures.npz")
SCANS = os.path.join(ROOT, "tests", "golden", "ref_scans.npz")
CLOUDS = ["sphere", "cube", "plane", "lattice", "dup"]
SCAN_NAMES = ["stanford_bunny", "fandisk", "detergent", "spray"]
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "box_search_test.cpp")
LIBDIR = os.path.join(ROOT, "point-cloud-processing_b200", "lib")
F32 = np.float32


def boxes_around(xyz, nb, frac_lo, frac_hi, seed):
    """nb boxes centred on random points of the cloud, half-sides a random fraction of its extent"""
    rng = np.random.default_rng(seed)
    ext = float(np.max(xyz.max(0) - xyz.min(0)))
    c = xyz[rng.choice(len(xyz), nb)]
    h = (rng.uniform(frac_lo, frac_hi, (nb, 3)) * ext).astype(F32)
    return np.concatenate([c - h, c + h], 1).astype(F32)


def check_exact(ix, xyz, boxes, sample=None, indexed=None):
    """unsorted and sorted search of every box; `sample`: the boxes checked against brute force
    (all when None).  Returns (offsets, unsorted idx)."""
    off, idx = ix.box_search(boxes)
    soff, sidx = ix.box_search(boxes, sorted=True)
    assert np.array_equal(off, soff)
    cnt = ix.box_count(boxes)
    assert np.array_equal(cnt, np.diff(off).astype(np.uint32))
    lists, slists = split_csr(off, idx), split_csr(soff, sidx)
    for a, b in zip(lists, slists):  # sorted == per-list np.sort of the unsorted result
        assert np.array_equal(np.sort(a), b)
    pick = range(len(boxes)) if sample is None else sample
    want = bruteforce_boxes(xyz, boxes[list(pick)], indexed)
    for w, b in zip(want, pick):
        assert np.array_equal(slists[b], w), (b, boxes[b], len(slists[b]), len(w))
    return off, idx


class _DeviceList:
    """a device list of uint32 seen by torch (read as int32, viewed back on the host)"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False),
                                         "version": 3, "strides": None}


def compile_cpp(pcpx, exe):
    pcpx.lib()  # the library must exist to link against
    subprocess.run(["g++", "-std=c++17", "-O2", "-Wall", "-Wextra", "-Werror",
                    "-I", os.path.join(ROOT, "include"), CPP_SRC, "-L", LIBDIR, "-lpcpx",
                    "-Wl,-rpath," + LIBDIR, "-o", str(exe)], check=True)


def test_dropin_box_overloads_compile(pcpx, tmp_path):
    exe = tmp_path / "box_search_test"
    compile_cpp(pcpx, exe)
    if pcpx.device_count() == 0:
        r = subprocess.run([str(exe)], capture_output=True, text=True)
        assert r.returncode == 2 and "no CPU path" in r.stderr


@pytest.mark.gpu
def test_dropin_box_overloads_match_contains(pcpx, tmp_path):
    exe = tmp_path / "box_search_test"
    compile_cpp(pcpx, exe)
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks hold" in r.stdout


@pytest.mark.gpu
@pytest.mark.parametrize("name", CLOUDS)
def test_reference_fixture_clouds(pcpx, name):
    xyz = np.load(FIX)[name + "_xyz"]
    boxes = np.concatenate([boxes_around(xyz, 300, 0.0, 0.05, 1), boxes_around(xyz, 100, 0.05, 0.4, 2),
                            np.array([[-np.inf] * 3 + [np.inf] * 3], F32)])
    with pcpx.Index(xyz) as ix:
        check_exact(ix, xyz, boxes)


@pytest.mark.gpu
@pytest.mark.parametrize("name", SCAN_NAMES)
def test_reference_scans(pcpx, name):
    xyz = np.load(SCANS)[name + "_xyz"]
    boxes = np.concatenate([boxes_around(xyz, 300, 0.0, 0.03, 3), boxes_around(xyz, 50, 0.03, 0.3, 4)])
    with pcpx.Index(xyz) as ix:
        check_exact(ix, xyz, boxes)


@pytest.mark.gpu
def test_uniform_cube_1m(pcpx):
    xyz = pcpx.synth.uniform_cube(1_000_000, half=100.0)
    # a cube of side s holds about 1e6 * (s / 200)^3 points: 0 .. ~1e4 for half-sides up to
    # 21.5 (boxes at the cloud's faces hold fewer)
    rng = np.random.default_rng(5)
    c = rng.uniform(-100, 100, (4096, 3)).astype(F32)
    h = (rng.uniform(0.0, 1.0, (4096, 1)) ** 2 * 21.5).astype(F32) * np.ones((1, 3), F32)
    boxes = np.concatenate([c - h, c + h], 1)
    with pcpx.Index(xyz) as ix:
        off, _ = check_exact(ix, xyz, boxes)
        cnt = np.diff(off)
        assert cnt.min() == 0 and 5_000 < cnt.max() < 20_000


@pytest.mark.gpu
def test_edge_cases(pcpx):
    xyz = pcpx.synth.uniform_cube(50_000, half=1.0)
    xyz = np.concatenate([xyz, np.repeat(xyz[:3], 3, axis=0)])
    inf, nan = np.inf, np.nan
    p = xyz[0]
    boxes = np.array([np.concatenate([p, p]), [-0.5, 0.5, -0.5, 0.5, -0.5, 0.5],
                      [nan, -1, -1, 1, 1, 1], [-1, -1, -1, 1, 1, nan], [-inf] * 3 + [inf] * 3,
                      [-inf, -0.1, -inf, inf, 0.1, inf], [2, 2, 2, 3, 3, 3], [-5] * 3 + [5] * 3,
                      [-inf] * 6, [inf] * 6], F32)
    with pcpx.Index(xyz) as ix:
        off, _ = check_exact(ix, xyz, boxes)
        cnt = np.diff(off)
        assert cnt[0] == 4 and cnt[1] == cnt[2] == cnt[3] == 0 and cnt[4] == cnt[7] == len(xyz)
        # no boxes
        off, idx = ix.box_search(np.zeros((0, 6), F32))
        assert off.tolist() == [0] and len(idx) == 0
        assert len(ix.box_count(np.zeros((0, 6), F32))) == 0
        # argument checks
        L = pcpx.lib()
        o = np.zeros(2, np.uint64)
        ptr = C.c_void_p()
        assert L.pcpx_box_search(ix._h, boxes.ctypes.data, 1, 20, o.ctypes.data, C.byref(ptr), 0) != 0
        assert L.pcpx_box_search(ix._h, boxes.ctypes.data, 1, 24, None, C.byref(ptr), 0) != 0
        assert L.pcpx_box_count(ix._h, boxes.ctypes.data, 1, 24, None) != 0
        assert L.pcpx_box_count(ix._h, boxes.ctypes.data, 1, 0, o.ctypes.data) != 0
    # an empty cloud
    with pcpx.Index(np.zeros((0, 3), F32)) as ix:
        off, idx = ix.box_search(boxes)
        assert off.tolist() == [0] * (len(boxes) + 1) and len(idx) == 0


@pytest.mark.gpu
def test_voxel_grid_and_offset_cloud(pcpx):
    xyz = pcpx.synth.uniform_cube(200_000, half=1.0)
    grid = ([-0.5, -0.6, -0.7], [0.5, 0.6, 0.4])
    indexed = np.all((xyz >= F32(grid[0])) & (xyz <= F32(grid[1])), axis=1)
    boxes = np.concatenate([boxes_around(xyz, 500, 0.0, 0.3, 6),
                            np.array([[-np.inf] * 3 + [np.inf] * 3], F32)])
    with pcpx.Index(xyz, voxel_grid=grid) as ix:
        off, _ = check_exact(ix, xyz, boxes, indexed=indexed)
        assert off[-1] - off[-2] == indexed.sum()
    far = (xyz + F32(1000.0)).astype(F32)
    with pcpx.Index(far) as ix:
        check_exact(ix, far, boxes_around(far, 500, 0.0, 0.1, 7))


@pytest.mark.gpu
def test_10m_plane(pcpx):
    xyz = pcpx.synth.noisy_plane(10_000_000)
    L = pcpx.synth.plane_extent(10_000_000)
    rng = np.random.default_rng(8)
    c = np.concatenate([rng.uniform(0, L, (65536, 2)), np.zeros((65536, 1))], 1).astype(F32)
    h = np.array([0.01, 0.01, 0.01], F32)
    small = np.concatenate([c - h, c + h], 1).astype(F32)
    with pcpx.Index(xyz) as ix:
        off, idx = ix.box_search(small)
        cnt = ix.box_count(small)
        assert np.array_equal(cnt, np.diff(off).astype(np.uint32))
        assert 20 < cnt.mean() < 60
        sample = np.sort(rng.choice(65536, 256, replace=False))
        want = bruteforce_boxes(xyz, small[sample])
        lists = split_csr(off, idx)
        for w, b in zip(want, sample):
            assert np.array_equal(np.sort(lists[b]), w)
        soff, sidx = ix.box_search(small, sorted=True)
        assert np.array_equal(soff, off)
        for a, b in zip(lists, split_csr(soff, sidx)):
            assert np.array_equal(np.sort(a), b)
        big = np.array([[0.3 * L, -1, -1, 0.31 * L, L + 1, 1],     # 1 % slab
                        [-1, -1, -1, 0.5 * L, L + 1, 1],           # half the cloud
                        [-np.inf] * 3 + [np.inf] * 3], F32)        # all of it
        off, _ = check_exact(ix, xyz, big)
        assert np.diff(off)[2] == len(xyz)
        _, sidx = ix.box_search(big[2:], sorted=True)
        assert np.array_equal(sidx, np.arange(len(xyz), dtype=np.uint32))


@pytest.mark.gpu
def test_identical_bytes_across_buffers_and_handles(pcpx):
    import torch

    xyz = pcpx.synth.noise_mix(300_000, seed=3)
    boxes = np.concatenate([boxes_around(xyz, 3000, 0.0, 0.02, 9), boxes_around(xyz, 20, 0.1, 0.5, 10)])
    nb = len(boxes)
    L = pcpx.lib()
    with pcpx.Index(xyz) as ix:
        h_off, h_idx = ix.box_search(boxes)
        h_cnt = ix.box_count(boxes)
        d_cnt = ix.box_count(torch.from_numpy(boxes).cuda())
        assert np.array_equal(d_cnt.cpu().numpy().astype(np.uint32), h_cnt)
        # host, device and strided (32-byte records) box buffers; host and device output
        b8 = np.zeros((nb, 8), F32)
        b8[:, :6] = boxes
        srcs = [(boxes, 24), (torch.from_numpy(boxes).cuda(), 24), (b8, 32),
                (torch.from_numpy(b8).cuda(), 32)]
        for src, stride in srcs:
            bptr = src.ctypes.data if isinstance(src, np.ndarray) else src.data_ptr()
            for flags in (0, 1):
                off = np.zeros(nb + 1, np.uint64)
                p = C.c_void_p()
                assert L.pcpx_box_search(ix._h, bptr, nb, stride, off.ctypes.data, C.byref(p),
                                         flags) == 0
                total = int(off[-1])
                if flags & 1:
                    got = torch.as_tensor(_DeviceList(p.value, total), device="cuda").cpu()
                    got = got.numpy().view(np.uint32)
                    L.pcpx_free(p, 1)
                else:
                    got = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)),
                                                shape=(max(total, 1),))[:total].copy()
                    L.pcpx_free(p, 0)
                assert np.array_equal(off, h_off) and np.array_equal(got, h_idx)
        t = ix.timings()
        assert t["kernel_launches"] >= 5
    os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"] = "1"
    try:
        with pcpx.Index(xyz, devices=[0, 0]) as many:
            m_off, m_idx = many.box_search(boxes)
            assert np.array_equal(m_off, h_off) and np.array_equal(m_idx, h_idx)
    finally:
        del os.environ["PCPX_TEST_SAME_DEVICE_REPLICAS"]


@pytest.mark.gpu
def test_concurrent_calls_from_host_threads(pcpx):
    xyz = pcpx.synth.noisy_plane(500_000, extent=2.0)
    sets = [boxes_around(xyz, 2000, 0.0, 0.01 * (i + 1), 20 + i) for i in range(4)]
    with pcpx.Index(xyz) as ix:
        want = [ix.box_search(b) for b in sets]
        got = [None] * 4
        errors = []

        def run(i):
            try:
                got[i] = ix.box_search(sets[i])
            except Exception as e:  # surfaced below
                errors.append(e)

        threads = [threading.Thread(target=run, args=(i,)) for i in range(4)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors
        for g, w in zip(got, want):
            assert np.array_equal(g[0], w[0]) and np.array_equal(g[1], w[1])
