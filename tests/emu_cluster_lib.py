"""ctypes loader for tests/emu/libpcpx_emu_cluster.so — the emulated index of tests/emu/emu.cu
plus the steps of pcpx_cluster_by_density (cluster_core.cuh) run on the host — and the brute-force
DBSCAN both the CPU and the GPU suite compare with.

TEST HARNESS ONLY: lets the CPU-only suite check the clustering against a brute force. It is not
a fallback of the product; libpcpx.so contains none of it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_lib import CSRC, EMU_DIR, ROOT, _f32, _f32p, _ptr, _u8p, _u32p

CLUSTER_SRC = os.path.join(EMU_DIR, "emu_cluster.cu")
CLUSTER_SO = os.path.join(EMU_DIR, "libpcpx_emu_cluster.so")
NOISE = 0xFFFFFFFF
F32 = np.float32


def build_cluster_emu(force=False):
    srcs = [CLUSTER_SRC, os.path.join(EMU_DIR, "emu.cu")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp"))
    ]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(CLUSTER_SO) or os.path.getmtime(CLUSTER_SO) < newest:
        subprocess.run(
            ["nvcc", "-std=c++17", "-O2", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013",
             "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
             "-I", os.path.join(ROOT, "include"), "-I", CSRC, CLUSTER_SRC, "-o", CLUSTER_SO],
            check=True, capture_output=True)


class ClusterEmu:
    def __init__(self):
        build_cluster_emu()
        L = C.CDLL(CLUSTER_SO)
        L.emu_index_create.restype = C.c_void_p
        L.emu_index_create.argtypes = [_f32p, C.c_size_t, C.c_int, _f32p, C.c_uint32, C.c_uint32]
        L.emu_index_destroy.argtypes = [C.c_void_p]
        L.emu_cluster.restype = C.c_uint64
        L.emu_cluster.argtypes = [C.c_void_p, C.c_float, C.c_uint32, _u32p, _u8p]
        self.L = L

    def cluster(self, xyz, r, min_points, voxel_grid=None):
        """(labels, n_clusters, core flags) of the emulated call"""
        xyz = _f32(xyz).reshape(-1, 3)
        n = len(xyz)
        vox = None if voxel_grid is None else _f32(np.concatenate(voxel_grid))
        h = self.L.emu_index_create(_ptr(xyz, _f32p), n, 0 if vox is None else 1,
                                    _ptr(vox, _f32p), 0, 0)
        try:
            labels = np.zeros(max(n, 1), np.uint32)
            core = np.zeros(max(n, 1), np.uint8)
            nc = self.L.emu_cluster(h, F32(r), int(min_points), _ptr(labels, _u32p),
                                    _ptr(core, _u8p))
        finally:
            self.L.emu_index_destroy(h)
        return labels[:n], int(nc), core[:n].astype(bool)


def ball_pairs(xyz, r, indexed=None):
    """every ordered pair (i, j), i != j, of indexed points with the library's fp32 predicate
    ((dx*dx)+(dy*dy))+(dz*dz) <= fl(r*r); candidates from a kd-tree at a slightly inflated radius"""
    from scipy.spatial import cKDTree

    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    ids = np.arange(len(xyz)) if indexed is None else np.nonzero(indexed)[0]
    rr = F32(r) * F32(r)
    if len(ids) == 0:
        e = np.zeros(0, np.int64)
        return e, e, np.zeros(0, F32)
    p = xyz[ids].astype(np.float64)
    reach = float(np.sqrt(float(rr))) * (1 + 1e-5) + 4 * float(np.spacing(F32(np.abs(p).max())))
    pairs = cKDTree(p).query_pairs(reach, output_type="ndarray")
    i, j = ids[pairs[:, 0]], ids[pairs[:, 1]]
    d = xyz[i] - xyz[j]  # fp32 differences: fl(a - b), negation-symmetric
    d2 = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    keep = d2 <= rr
    i, j, d2 = i[keep], j[keep], d2[keep]
    return np.concatenate([i, j]), np.concatenate([j, i]), np.concatenate([d2, d2])


def bruteforce_dbscan(xyz, r, min_points, indexed=None, pairs=None):
    """(labels, n_clusters, core) by the contract of pcpx_cluster_by_density: core iff the ball
    (itself included) holds >= min_points indexed points; clusters = connected_components of the
    core subgraph, numbered by smallest original index; border = the core neighbour with the
    smallest (d2, index); noise otherwise.  pairs: ball_pairs(...) when already computed."""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    xyz = np.asarray(xyz, F32).reshape(-1, 3)
    n = len(xyz)
    idx_mask = np.ones(n, bool) if indexed is None else np.asarray(indexed, bool)
    i, j, d2 = ball_pairs(xyz, r, idx_mask) if pairs is None else pairs
    count = np.bincount(i, minlength=n) + idx_mask  # + the point itself
    core = idx_mask & (count >= min_points)
    labels = np.full(n, NOISE, np.uint32)
    cids = np.nonzero(core)[0]
    n_clusters = 0
    if len(cids):
        pos = np.full(n, -1, np.int64)
        pos[cids] = np.arange(len(cids))
        e = core[i] & core[j]
        g = coo_matrix((np.ones(int(e.sum()), np.int8), (pos[i[e]], pos[j[e]])),
                       shape=(len(cids), len(cids)))
        n_clusters, comp = connected_components(g, directed=False)
        # connected_components numbers components by their smallest vertex, as the contract does
        labels[cids] = comp.astype(np.uint32)
    # border points: among core neighbours, the smallest (d2, index)
    b = idx_mask[i] & ~core[i] & core[j]
    if b.any():
        bi, bj, bd = i[b], j[b], d2[b]
        order = np.lexsort((bj, bd, bi))
        bi, bj = bi[order], bj[order]
        firsts = np.ones(len(bi), bool)
        firsts[1:] = bi[1:] != bi[:-1]
        labels[bi[firsts]] = labels[bj[firsts]]
    return labels, int(n_clusters), core
