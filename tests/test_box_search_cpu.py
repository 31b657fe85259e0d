"""Axis-aligned box range search (pcpx_box_search) without a GPU: the device traversal
(box_visit in box_core.cuh, run on the host by the emulation library) against a numpy brute force
of the fp32 predicate min <= p <= max.  Comparisons only, no arithmetic: every box's list must be
set-exact."""
import numpy as np
import pytest

from emu_box_lib import bruteforce_boxes, split_csr

F32 = np.float32


@pytest.fixture(scope="module")
def box_emu():
    from emu_box_lib import BoxEmu

    return BoxEmu()


def check(box_emu, xyz, boxes, voxel_grid=None, max_level=0):
    """every box exact; returns the emulated (offsets, idx, spans)"""
    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    boxes = np.asarray(boxes, F32).reshape(-1, 6)
    ix = box_emu.index(xyz, voxel_grid=voxel_grid, max_level=max_level)
    off, idx, spans = ix.box_search(boxes)
    indexed = None
    if voxel_grid is not None:
        lo, hi = (np.asarray(v, F32) for v in voxel_grid)
        indexed = np.all((xyz >= lo) & (xyz <= hi), axis=1)
    want = bruteforce_boxes(xyz, boxes, indexed)
    assert len(off) == len(boxes) + 1
    for b, (got, w) in enumerate(zip(split_csr(off, idx), want)):
        assert np.array_equal(np.sort(got), w), (b, boxes[b], len(got), len(w))
    return off, idx, spans


def lattice(m, spacing, origin=0.0):
    g = np.arange(m, dtype=np.float64) * spacing + origin
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3).astype(F32)


def faces_and_ulps(values, rng, nb):
    """boxes whose faces are the given planes, or one ulp either side of them"""
    v = np.asarray(values, F32)
    out = []
    for _ in range(nb):
        lo = rng.choice(v, 3)
        hi = rng.choice(v, 3)
        lo, hi = np.minimum(lo, hi), np.maximum(lo, hi)
        for a in range(3):
            lo[a] = [lo[a], np.nextafter(lo[a], F32(-np.inf)), np.nextafter(lo[a], F32(np.inf))][rng.integers(3)]
            hi[a] = [hi[a], np.nextafter(hi[a], F32(-np.inf)), np.nextafter(hi[a], F32(np.inf))][rng.integers(3)]
        out.append(np.concatenate([lo, hi]))
    return np.array(out, F32)


def test_reference_range_scenario(box_emu):
    # test/octree/octree_range_search.cpp, as restated by tests/cpp/dropin_test.cpp
    pts = []
    for z in (-1.0, 1.0):
        for x, y in ((-1, -1), (1, -1), (1, 1), (-1, 1)):
            pts += [(0.5 * x, 0.5 * y, 0.5 * z), (0.4 * x, 0.3 * y, 0.6 * z)]
    pts = np.array(pts, F32)
    boxes = [[1.05, 1.05, 1.05, 2, 2, 2], [-2, -2, -2, 0, 0, 0]]
    off, idx, _ = check(box_emu, pts, boxes, voxel_grid=([-1] * 3, [1] * 3))
    assert np.diff(off).tolist() == [0, 2]
    assert sorted(idx.tolist()) == [0, 1]


@pytest.mark.parametrize("voxel", [False, True])
def test_power_of_two_lattice_on_cell_faces(box_emu, voxel):
    # root cube of side E = fp32(1 * 1.0001) over the voxel grid [0, 1]^3: a spacing of E / 16
    # puts the lattice planes on the nominal cell faces of levels 0..4
    E = float(F32(F32(1.0) * F32(1.0001)))
    xyz = lattice(16, E / 16)
    rng = np.random.default_rng(1)
    # the planes themselves plus points one ulp either side of some of them
    jit = xyz[rng.choice(len(xyz), 400, replace=False)].copy()
    jit[:200] = np.nextafter(jit[:200], F32(np.inf))
    jit[200:] = np.nextafter(jit[200:], F32(-np.inf))
    xyz = np.concatenate([xyz, jit])
    planes = np.unique(lattice(16, E / 16)[:, 0])
    boxes = faces_and_ulps(planes, rng, 600)
    grid = ([0, 0, 0], [1, 1, 1]) if voxel else None
    _, _, spans = check(box_emu, xyz, boxes, voxel_grid=grid)
    assert spans.sum() > 0  # INSIDE cells were emitted whole


@pytest.mark.parametrize("max_level", [0, 2, 12])
def test_lattice_at_forced_levels(box_emu, max_level):
    xyz = lattice(20, 0.125, origin=-1.0)
    rng = np.random.default_rng(2)
    planes = np.unique(xyz[:, 0])
    boxes = np.concatenate([faces_and_ulps(planes, rng, 300),
                            np.sort(rng.uniform(-1.2, 1.5, (200, 2, 3)).astype(F32), axis=1).reshape(-1, 6)])
    check(box_emu, xyz, boxes, max_level=max_level)


def test_far_lattice(box_emu):
    # dropin_test.cpp: 9 x 9 x 9 lattice of spacing 1e-4 near x = y = z = 100
    g = (F32(100.0) + F32(1e-4) * np.arange(9, dtype=F32)).astype(F32)
    xyz = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3).astype(F32)
    box = np.concatenate([xyz[(2 * 9 + 2) * 9 + 2], xyz[(6 * 9 + 6) * 9 + 6]])
    rng = np.random.default_rng(3)
    off, _, _ = check(box_emu, xyz, np.concatenate([box[None], faces_and_ulps(g, rng, 300)]))
    assert off[1] >= 125


def test_cloud_offset_by_1e3(box_emu, pcpx):
    xyz = (pcpx.synth.uniform_cube(20000, half=1.0) + F32(1000.0)).astype(F32)
    rng = np.random.default_rng(4)
    c = xyz[rng.choice(len(xyz), 300)]
    h = rng.uniform(0.0, 0.3, (300, 3)).astype(F32)
    boxes = np.concatenate([c - h, c + h], axis=1)
    off, _, _ = check(box_emu, xyz, boxes)
    assert np.diff(off).max() > 100


def test_degenerate_boxes(box_emu, pcpx):
    rng = np.random.default_rng(5)
    xyz = pcpx.synth.uniform_cube(5000, half=1.0)
    xyz = np.concatenate([xyz, np.repeat(xyz[:5], 4, axis=0)])  # duplicated points
    p, d = xyz[17], xyz[3]
    inf, nan = np.inf, np.nan
    boxes = [
        np.concatenate([p, p]),                      # zero volume on a point
        np.concatenate([d, d]),                      # ... on a point held five times
        [-0.5, 0.5, -0.5, 0.5, -0.5, 0.5],           # min > max on y
        [-0.5, -0.5, -0.5, 0.5, 0.5, 0.5],
        [nan, -0.5, -0.5, 0.5, 0.5, 0.5],            # NaN bounds
        [-0.5, -0.5, -0.5, 0.5, nan, 0.5],
        [-inf, -inf, -inf, inf, inf, inf],           # everything
        [-inf, -0.2, -inf, inf, 0.2, inf],
        [0.1, -inf, -inf, inf, inf, inf],
        [inf, inf, inf, inf, inf, inf],
        [-inf, -inf, -inf, -inf, -inf, -inf],
        [2.0, 2.0, 2.0, 3.0, 3.0, 3.0],              # wholly outside the root voxel
        [-3.0, -3.0, -3.0, -2.0, 3.0, 3.0],
        [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0],           # the whole cloud
        [-5.0, -5.0, -5.0, 5.0, 5.0, 5.0],
    ]
    off, _, spans = check(box_emu, xyz, np.array(boxes, F32))
    cnt = np.diff(off)
    assert cnt[0] == 1 and cnt[1] == 5
    assert cnt[2] == 0 and cnt[4] == 0 and cnt[5] == 0
    assert cnt[6] == len(xyz) and cnt[14] == len(xyz)
    assert spans[6] <= 8 and spans[14] <= 8  # a box over the whole cloud is a few whole spans


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_thin_slabs(box_emu, pcpx, axis):
    xyz = pcpx.synth.uniform_cube(30000, half=1.0)
    rng = np.random.default_rng(6 + axis)
    boxes = []
    for t in (1e-3, 1e-2, 0.05):
        for c in rng.uniform(-1, 1, 20):
            b = np.array([-2, -2, -2, 2, 2, 2], F32)
            b[axis], b[3 + axis] = c - t, c + t
            boxes.append(b)
    check(box_emu, xyz, np.array(boxes, F32))


def test_voxel_grid_excludes_points_inside_the_box(box_emu, pcpx):
    xyz = pcpx.synth.uniform_cube(20000, half=1.0)
    grid = ([-0.5, -0.6, -0.7], [0.5, 0.6, 0.4])
    rng = np.random.default_rng(8)
    c = rng.uniform(-1, 1, (200, 3)).astype(F32)
    h = rng.uniform(0.05, 0.8, (200, 3)).astype(F32)
    boxes = np.concatenate([np.concatenate([c - h, c + h], 1),
                            np.array([[-1, -1, -1, 1, 1, 1], [-np.inf] * 3 + [np.inf] * 3], F32)])
    off, _, _ = check(box_emu, xyz, boxes, voxel_grid=grid)
    inside = np.all((xyz >= np.float32(grid[0])) & (xyz <= np.float32(grid[1])), axis=1)
    assert off[-1] - off[-2] == inside.sum() < len(xyz)


def test_surfaces_and_big_leaves(box_emu, pcpx):
    rng = np.random.default_rng(9)
    for xyz in (pcpx.synth.noisy_plane(30000, extent=1.0), pcpx.synth.noisy_sphere(30000)):
        c = xyz[rng.choice(len(xyz), 300)]
        h = rng.uniform(0.001, 0.2, (300, 3)).astype(F32)
        check(box_emu, xyz, np.concatenate([c - h, c + h], 1))
    # one fine cell holding 500 copies of a point: a PARTIAL leaf of more than 32 points
    xyz = np.concatenate([pcpx.synth.uniform_cube(3000, half=1.0), np.full((500, 3), 0.25, F32)])
    boxes = np.array([[0.25, 0.25, 0.25, 0.25, 0.25, 0.25], [0.2, 0.2, 0.2, 0.25, 0.3, 0.3],
                      [0.2500001, 0.2, 0.2, 0.3, 0.3, 0.3]], F32)
    off, _, _ = check(box_emu, xyz, boxes)
    assert np.diff(off)[0] == 500 and np.diff(off)[2] < 500


def test_empty_cloud_and_no_boxes(box_emu, pcpx):
    off, idx, _ = check(box_emu, np.zeros((0, 3), F32), [[-1, -1, -1, 1, 1, 1]])
    assert off.tolist() == [0, 0] and len(idx) == 0
    off, idx, _ = check(box_emu, pcpx.synth.uniform_cube(100, half=1.0), np.zeros((0, 6), F32))
    assert off.tolist() == [0] and len(idx) == 0


def test_fill_order_is_a_permutation_of_the_set(box_emu, pcpx):
    xyz = pcpx.synth.noisy_plane(20000, extent=1.0)
    rng = np.random.default_rng(10)
    c = xyz[rng.choice(len(xyz), 100)]
    h = rng.uniform(0.01, 0.5, (100, 3)).astype(F32)
    off, idx, _ = check(box_emu, xyz, np.concatenate([c - h, c + h], 1))
    for lst in split_csr(off, idx):
        assert len(np.unique(lst)) == len(lst)
    # deterministic: the same call gives the same bytes
    ix = box_emu.index(xyz)
    a = ix.box_search(np.concatenate([c - h, c + h], 1))
    b = ix.box_search(np.concatenate([c - h, c + h], 1))
    assert np.array_equal(a[1], b[1])
