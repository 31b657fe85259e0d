"""ctypes loader for tests/emu/libpcpx_emu_icp.so — the emulated index of tests/emu/emu.cu plus
the correspondence pass, the host solve and the loop of pcpx_icp (icp_core.cuh, icp_solve.hpp) run
on the host — and the numpy references both the CPU and the GPU suite compare with: the
brute-force bounded nearest neighbour, the fp64 normal equations and the solve.

TEST HARNESS ONLY: lets the CPU-only suite check the registration against a brute force. It is
not a fallback of the product; libpcpx.so contains none of it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_lib import CSRC, EMU_DIR, ROOT, _f32, _f32p, _ptr, _u32p, _u64p

ICP_SRC = os.path.join(EMU_DIR, "emu_icp.cu")
ICP_SO = os.path.join(EMU_DIR, "libpcpx_emu_icp.so")
NONE = 0xFFFFFFFF
F32 = np.float32
_f64p = C.POINTER(C.c_double)
N_TERMS = {0: 29, 1: 17}


def build_icp_emu(force=False):
    srcs = [ICP_SRC, os.path.join(EMU_DIR, "emu.cu")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp"))
    ]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(ICP_SO) or os.path.getmtime(ICP_SO) < newest:
        subprocess.run(
            ["nvcc", "-std=c++17", "-O2", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013",
             "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
             "-I", os.path.join(ROOT, "include"), "-I", CSRC, ICP_SRC, "-o", ICP_SO],
            check=True, capture_output=True)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


class IcpEmu:
    def __init__(self):
        build_icp_emu()
        L = C.CDLL(ICP_SO)
        L.emu_index_create.restype = C.c_void_p
        L.emu_index_create.argtypes = [_f32p, C.c_size_t, C.c_int, _f32p, C.c_uint32, C.c_uint32]
        L.emu_index_destroy.argtypes = [C.c_void_p]
        L.emu_nearest_within.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f64p, C.c_float, _u32p,
                                         _f32p]
        L.emu_icp_sums.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f64p, C.c_float, C.c_uint32,
                                   _f32p, _f64p, _f64p, _u32p]
        L.emu_icp_solve.argtypes = [C.c_uint32, _f64p, _f64p]
        L.emu_icp_update.argtypes = [_f64p, _f64p, _f64p]
        L.emu_icp.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_uint32, C.c_uint32,
                              C.c_float, C.c_double, C.c_double, _f64p, _f64p, _u64p, _u32p]
        self.L = L

    def index(self, xyz, voxel_grid=None):
        return _EmuIndex(self.L, xyz, voxel_grid)

    def solve(self, metric, sums):
        x = np.zeros(6)
        self.L.emu_icp_solve(metric, _ptr(_f64(sums), _f64p), _ptr(x, _f64p))
        return x

    def update(self, T, x, c):
        T = _f64(T).reshape(4, 4).copy()
        self.L.emu_icp_update(_ptr(T, _f64p), _ptr(_f64(x), _f64p), _ptr(_f64(c), _f64p))
        return T


class _EmuIndex:
    def __init__(self, L, xyz, voxel_grid):
        self.L = L
        self.xyz = _f32(xyz).reshape(-1, 3)
        vox = None if voxel_grid is None else _f32(np.concatenate(voxel_grid))
        self.h = L.emu_index_create(_ptr(self.xyz, _f32p), len(self.xyz),
                                    0 if vox is None else 1, _ptr(vox, _f32p), 0, 0)
        if voxel_grid is not None:
            lo, hi = voxel_grid
        elif len(self.xyz):
            lo, hi = self.xyz.min(0), self.xyz.max(0)
        else:
            lo = hi = np.zeros(3, F32)
        lo, hi = np.asarray(lo, F32).astype(np.float64), np.asarray(hi, F32).astype(np.float64)
        self.centre = 0.5 * (lo + hi)

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.L.emu_index_destroy(self.h)

    def nearest_within(self, q, r, T=None):
        q = _f32(q).reshape(-1, 3)
        idx = np.zeros(max(len(q), 1), np.uint32)
        d2 = np.zeros(max(len(q), 1), F32)
        self.L.emu_nearest_within(self.h, _ptr(q, _f32p), len(q), _ptr(_f64(T), _f64p), F32(r),
                                  _ptr(idx, _u32p), _ptr(d2, _f32p))
        return idx[:len(q)], d2[:len(q)]

    def sums(self, src, r, metric, T=None, normals=None):
        src = _f32(src).reshape(-1, 3)
        T = np.eye(4) if T is None else T
        s = np.zeros(29)
        corr = np.zeros(max(len(src), 1), np.uint32)
        self.L.emu_icp_sums(self.h, _ptr(src, _f32p), len(src), _ptr(_f64(T), _f64p), F32(r),
                            metric, _ptr(_f32(normals), _f32p), _ptr(self.centre, _f64p),
                            _ptr(s, _f64p), _ptr(corr, _u32p))
        return s[:N_TERMS[metric]], corr[:len(src)]

    def icp(self, src, r, metric, normals=None, init=None, max_it=30, rot_tol=1e-6,
            trans_tol=None):
        src = _f32(src).reshape(-1, 3)
        if trans_tol is None:
            lo, hi = self.xyz.min(0).astype(np.float64), self.xyz.max(0).astype(np.float64)
            trans_tol = 1e-6 * float(np.linalg.norm(hi - lo))
        T = np.eye(4) if init is None else _f64(init).reshape(4, 4).copy()
        out3 = np.zeros(3, np.uint64)
        corr = np.zeros(max(len(src), 1), np.uint32)
        self.L.emu_icp(self.h, _ptr(src, _f32p), len(src), _ptr(_f32(normals), _f32p), metric,
                       max_it, F32(r), rot_tol, trans_tol, _ptr(self.centre, _f64p),
                       _ptr(T, _f64p), _ptr(out3, _u64p), _ptr(corr, _u32p))
        return T, [int(v) for v in out3], corr[:len(src)]


# ---- numpy references ------------------------------------------------------------------------

def transform_f32(q, T):
    """y = ((R0 x + R1 y) + R2 z) + t per component in fp64 (numpy never fuses), rounded once"""
    q = np.asarray(q, F32).reshape(-1, 3).astype(np.float64)
    T = np.asarray(T, np.float64).reshape(4, 4)
    y = np.empty_like(q)
    for a in range(3):
        y[:, a] = ((T[a, 0] * q[:, 0] + T[a, 1] * q[:, 1]) + T[a, 2] * q[:, 2]) + T[a, 3]
    return y.astype(F32)


def sqdist_f32(a, b):
    d = np.asarray(a, F32) - np.asarray(b, F32)
    return (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]


def brute_nearest_within(target, y, r, indexed=None):
    """(idx, d2) by the contract of pcpx_nearest_within: the indexed point with the smallest
    (fp32 no-FMA d2, index) among those with d2 <= fl(r * r); candidates from a kd-tree ball
    slightly beyond the fp64 nearest distance, so no fp32 tie or rounding can be missed"""
    from scipy.spatial import cKDTree

    target = np.asarray(target, F32).reshape(-1, 3)
    y = np.asarray(y, F32).reshape(-1, 3)
    n = len(y)
    idx = np.full(n, NONE, np.uint32)
    d2 = np.full(n, np.inf, F32)
    ids = np.arange(len(target)) if indexed is None else np.nonzero(indexed)[0]
    fin = np.all(np.isfinite(y), axis=1)
    if len(ids) == 0 or not fin.any():
        return idx, d2
    rr = F32(r) * F32(r)
    pts = target[ids].astype(np.float64)
    tree = cKDTree(pts)
    qi = np.nonzero(fin)[0]
    yd = y[qi].astype(np.float64)
    dist, _ = tree.query(yd, k=1)
    scale = max(float(np.abs(pts).max()), float(np.abs(yd).max()), 1e-30)
    reach = dist * (1 + 1e-5) + 8 * float(np.spacing(F32(scale)))
    ok = dist <= np.sqrt(float(rr)) * (1 + 1e-5) + 8 * float(np.spacing(F32(scale)))
    qi, yd, reach = qi[ok], yd[ok], reach[ok]
    if len(qi) == 0:
        return idx, d2
    lists = tree.query_ball_point(yd, reach, return_sorted=False)
    lens = np.array([len(l) for l in lists])
    rows = np.repeat(qi, lens)
    cand = ids[np.concatenate([np.asarray(l, np.int64) for l in lists])]
    cd2 = sqdist_f32(target[cand], y[rows])
    keep = cd2 <= rr
    rows, cand, cd2 = rows[keep], cand[keep], cd2[keep]
    order = np.lexsort((cand, cd2, rows))
    rows, cand, cd2 = rows[order], cand[order], cd2[order]
    first = np.ones(len(rows), bool)
    first[1:] = rows[1:] != rows[:-1]
    idx[rows[first]] = cand[first]
    d2[rows[first]] = cd2[first]
    return idx, d2


def np_sums(metric, y, q, d2, c, n=None):
    """the reduced sums (layout of icp_solve.hpp) over the pairs (y_i, q_i) in fp64"""
    y = np.asarray(y, F32).astype(np.float64)
    q = np.asarray(q, F32).astype(np.float64)
    c = np.asarray(c, np.float64)
    py, pq = y - c, q - c
    if metric == 0:
        n = np.asarray(n, F32).astype(np.float64)
        J = np.concatenate([np.cross(py, n), n], axis=1)
        r = ((y - q) * n).sum(1)
        A = J.T @ J
        iu = np.triu_indices(6)
        return np.concatenate([A[iu], J.T @ r, [np.sum(np.asarray(d2, np.float64)), len(y)]])
    M = py.T @ pq
    return np.concatenate([py.sum(0), pq.sum(0), M.reshape(9),
                           [np.sum(np.asarray(d2, np.float64)), len(y)]])


def np_solve(metric, s):
    """the step (omega, v): eigh pseudo-inverse (plane) or SVD Kabsch (point)"""
    from scipy.spatial.transform import Rotation

    s = np.asarray(s, np.float64)
    if metric == 0:
        A = np.zeros((6, 6))
        A[np.triu_indices(6)] = s[:21]
        A = A + np.triu(A, 1).T
        w, V = np.linalg.eigh(A)
        keep = w > 1e-12 * w.max()
        return -(V[:, keep] / w[keep]) @ (V[:, keep].T @ s[21:27])
    n = s[16]
    my, mq = s[0:3] / n, s[3:6] / n
    S = s[6:15].reshape(3, 3) - n * np.outer(my, mq)
    U, _, Vt = np.linalg.svd(S)
    D = np.diag([1.0, 1.0, np.sign(np.linalg.det(Vt.T @ U.T))])
    R = Vt.T @ D @ U.T
    return np.concatenate([Rotation.from_matrix(R).as_rotvec(), mq - R @ my])


def np_update(T, x, c):
    from scipy.spatial.transform import Rotation

    R = Rotation.from_rotvec(x[:3]).as_matrix()
    U = np.eye(4)
    U[:3, :3] = R
    U[:3, 3] = np.asarray(c) + x[3:] - R @ np.asarray(c)
    return U @ np.asarray(T, np.float64).reshape(4, 4)


def np_step(metric, target, normals, src, r, T, c, indexed=None):
    """one ICP step by the contract: brute-force pairs under T, fp64 sums, numpy solve; returns
    (T', sums)"""
    y = transform_f32(src, T)
    idx, d2 = brute_nearest_within(target, y, r, indexed)
    ok = idx != NONE
    if metric == 0:
        nn = np.asarray(normals, F32)[idx[ok].astype(np.int64)]
        fin = np.all(np.isfinite(nn), axis=1)
        sel = np.nonzero(ok)[0][fin]
        s = np_sums(0, y[sel], target[idx[sel].astype(np.int64)], d2[sel], c, nn[fin])
    else:
        sel = np.nonzero(ok)[0]
        s = np_sums(1, y[sel], target[idx[sel].astype(np.int64)], d2[sel], c)
    return np_update(T, np_solve(metric, s), c), s


def rigid(angle_deg, axis, t):
    """4 x 4 rotation by angle_deg about axis, then translation t"""
    from scipy.spatial.transform import Rotation

    axis = np.asarray(axis, np.float64)
    T = np.eye(4)
    T[:3, :3] = Rotation.from_rotvec(np.deg2rad(angle_deg) * axis / np.linalg.norm(axis)).as_matrix()
    T[:3, 3] = t
    return T


def pose_error(T, T_ref):
    """(rotation angle in rad, translation distance) of T_ref^-1 T"""
    D = np.linalg.inv(np.asarray(T_ref)) @ np.asarray(T)
    ang = float(np.arccos(np.clip((np.trace(D[:3, :3]) - 1) / 2, -1, 1)))
    return ang, float(np.linalg.norm(D[:3, 3]))
