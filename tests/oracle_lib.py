"""ctypes loaders for the CPU checkers (TEST INFRASTRUCTURE — never used by the product).

* ``Oracle``   — oracle/liboracle.so, the plain-C restatement (oracle/pcp_oracle.c).
* ``RefBridge`` — oracle/_ref/libpcp_ref.so, the UNMODIFIED reference headers behind a flat C
  bridge (oracle/ref_bridge.cpp). Only buildable when the environment variable PCP_REFERENCE
  names a checkout of the reference (REFERENCE_DIR); a prebuilt oracle/_ref is used as it is.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_SO = os.path.join(ORACLE_DIR, "liboracle.so")
REF_SO = os.path.join(ORACLE_DIR, "_ref", "libpcp_ref.so")
REF_SMOOTHING_SO = os.path.join(ORACLE_DIR, "_ref", "libpcp_ref_smoothing.so")
REF_ORIENT_SO = os.path.join(ORACLE_DIR, "_ref", "libpcp_ref_orient.so")
REF_PLY_SO = os.path.join(ORACLE_DIR, "_ref", "libpcp_ref_ply.so")
REFERENCE_DIR = os.environ.get("PCP_REFERENCE") or None  # a checkout of Q-Minh/point-cloud-processing

_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_u8p = C.POINTER(C.c_uint8)


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(t)


def _f32(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float32)


def build_oracle(force=False):
    """Compile the checker libraries (make -C oracle). Building the checker is not using it."""
    src = os.path.join(ORACLE_DIR, "pcp_oracle.c")
    stale = (not os.path.exists(ORACLE_SO)) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(src)
    ref_possible = REFERENCE_DIR is not None and os.path.isdir(
        os.path.join(REFERENCE_DIR, "include", "pcp"))
    ref_src = os.path.join(ORACLE_DIR, "ref_bridge.cpp")
    ref_stale = ref_possible and (
        (not os.path.exists(REF_SO)) or os.path.getmtime(REF_SO) < os.path.getmtime(ref_src)
    )
    for so, name in ((REF_SMOOTHING_SO, "ref_bridge_smoothing.cpp"),
                     (REF_ORIENT_SO, "ref_bridge_orient.cpp"),
                     (REF_PLY_SO, "ref_bridge_ply.cpp")):
        bridge_src = os.path.join(ORACLE_DIR, name)
        ref_stale = ref_stale or (ref_possible and (
            (not os.path.exists(so)) or os.path.getmtime(so) < os.path.getmtime(bridge_src)))
    if force or stale or ref_stale:
        subprocess.run(["make", "-C", ORACLE_DIR, "all"], check=True, capture_output=True)


def nthreads_default():
    return max(1, os.cpu_count() or 1)


class Oracle:
    def __init__(self):
        build_oracle()
        L = C.CDLL(ORACLE_SO)
        L.oracle_cloud_create.restype = C.c_void_p
        L.oracle_cloud_create.argtypes = [_f32p, C.c_size_t, _f32p, C.c_uint32, C.c_uint32]
        L.oracle_cloud_destroy.argtypes = [C.c_void_p]
        L.oracle_cloud_size.restype = C.c_size_t
        L.oracle_cloud_size.argtypes = [C.c_void_p]
        L.oracle_cloud_nodes.restype = C.c_size_t
        L.oracle_cloud_nodes.argtypes = [C.c_void_p]
        L.oracle_cloud_bbox.argtypes = [C.c_void_p, _f32p]
        L.oracle_bounding_box.argtypes = [_f32p, C.c_size_t, _f32p]
        L.oracle_squared_distance.restype = C.c_float
        L.oracle_squared_distance.argtypes = [_f32p, _f32p]
        L.oracle_are_vectors_equal.restype = C.c_int
        L.oracle_are_vectors_equal.argtypes = [_f32p, _f32p, C.c_float]
        L.oracle_knn.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, C.c_double,
                                 _i64p, _f32p, _u32p, C.c_int]
        L.oracle_estimate_normals.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t,
                                              C.c_double, _f32p, _f32p, C.c_int]
        L.oracle_radius.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_float, C.c_int,
                                    _u32p, _u64p, _i64p, C.c_int]
        L.oracle_average_distance_to_neighbors.restype = C.c_float
        L.oracle_average_distance_to_neighbors.argtypes = [C.c_void_p, C.c_size_t, C.c_double,
                                                           _f32p, C.c_int]
        L.oracle_density_filter.restype = C.c_size_t
        L.oracle_density_filter.argtypes = [C.c_void_p, C.c_float, C.c_uint32, _u8p, _u32p,
                                            C.c_int]
        L.oracle_estimate_normal.argtypes = [_f32p, C.c_size_t, _f32p, _f32p]
        L.oracle_scatter_matrix.argtypes = [_f32p, C.c_size_t, _f32p, _f32p]
        L.oracle_knn_bruteforce.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t, C.c_size_t,
                                            C.c_double, _i64p, _f32p, _u32p]
        L.oracle_radius_count_bruteforce.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t,
                                                     _f32p, C.c_float, _u32p]
        _sz, _dbl = C.c_size_t, C.c_double
        L.oracle_bilateral_filter_points.argtypes = [_f32p, _f32p, _sz, _dbl, _dbl, _sz, _f32p]
        L.oracle_bilateral_filter_normals.argtypes = [_f32p, _f32p, _sz, _dbl, _dbl, _sz, _f32p]
        L.oracle_wlop.argtypes = [_f32p, _sz, _u32p, _sz, _dbl, _dbl, _sz, C.c_int, _f32p]
        L.oracle_propagate_normal_orientations.argtypes = [_f32p, _sz, _i64p, _sz, C.c_int, _f32p]
        self.L = L

    def propagate_normal_orientations(self, xyz, knn, normals, reverse_edges=True):
        """knn: n x k int64 neighbour indices, nearest first, -1 = none.  Returns a copy."""
        xyz = _f32(xyz).reshape(-1, 3)
        knn = np.ascontiguousarray(knn, dtype=np.int64)
        out = _f32(normals).reshape(-1, 3).copy()
        self.L.oracle_propagate_normal_orientations(_ptr(xyz, _f32p), len(xyz), _ptr(knn, _i64p),
                                                    knn.shape[1], 1 if reverse_edges else 0,
                                                    _ptr(out, _f32p))
        return out

    # ---- radius-search callers (SURVEY.md 8f rank 3) ---------------------------------------
    def bilateral_filter_points(self, xyz, normals, sigmaf, sigmag, iterations):
        xyz, normals = _f32(xyz).reshape(-1, 3), _f32(normals).reshape(-1, 3)
        out = np.zeros_like(xyz)
        self.L.oracle_bilateral_filter_points(_ptr(xyz, _f32p), _ptr(normals, _f32p), len(xyz),
                                              sigmaf, sigmag, iterations, _ptr(out, _f32p))
        return out

    def bilateral_filter_normals(self, xyz, normals, sigmaf, sigmag, iterations):
        xyz, normals = _f32(xyz).reshape(-1, 3), _f32(normals).reshape(-1, 3)
        out = np.zeros_like(xyz)
        self.L.oracle_bilateral_filter_normals(_ptr(xyz, _f32p), _ptr(normals, _f32p), len(xyz),
                                               sigmaf, sigmag, iterations, _ptr(out, _f32p))
        return out

    def wlop(self, xyz, initial, mu, h, iterations, uniform=True):
        xyz = _f32(xyz).reshape(-1, 3)
        initial = np.ascontiguousarray(initial, dtype=np.uint32)
        out = np.zeros((len(initial), 3), np.float32)
        self.L.oracle_wlop(_ptr(xyz, _f32p), len(xyz), _ptr(initial, _u32p), len(initial), mu, h,
                           iterations, 1 if uniform else 0, _ptr(out, _f32p))
        return out

    # ---- scalar helpers -----------------------------------------------------------------
    def squared_distance(self, a, b):
        a, b = _f32(a), _f32(b)
        return np.float32(self.L.oracle_squared_distance(_ptr(a, _f32p), _ptr(b, _f32p)))

    def are_vectors_equal(self, a, b, eps=1e-5):
        a, b = _f32(a), _f32(b)
        return bool(self.L.oracle_are_vectors_equal(_ptr(a, _f32p), _ptr(b, _f32p),
                                                    np.float32(eps)))

    def bounding_box(self, xyz):
        xyz = _f32(xyz)
        out = np.zeros(6, np.float32)
        self.L.oracle_bounding_box(_ptr(xyz, _f32p), len(xyz), _ptr(out, _f32p))
        return out

    def estimate_normal(self, pts):
        pts = _f32(pts).reshape(-1, 3)
        out = np.zeros(3, np.float32)
        gap = np.zeros(1, np.float32)
        self.L.oracle_estimate_normal(_ptr(pts, _f32p), len(pts), _ptr(out, _f32p),
                                      _ptr(gap, _f32p))
        return out, float(gap[0])

    def scatter_matrix(self, pts):
        pts = _f32(pts).reshape(-1, 3)
        c = np.zeros(6, np.float32)
        mu = np.zeros(3, np.float32)
        self.L.oracle_scatter_matrix(_ptr(pts, _f32p), len(pts), _ptr(c, _f32p), _ptr(mu, _f32p))
        return c, mu

    # ---- cloud --------------------------------------------------------------------------
    def cloud(self, xyz, bbox=None, node_capacity=0, max_depth=0):
        return OracleCloud(self, xyz, bbox, node_capacity, max_depth)

    def knn_bruteforce(self, xyz, queries, k, eps=1e-5):
        xyz = _f32(xyz)
        q = _f32(queries)
        nq = len(xyz) if q is None else len(q)
        idx = np.full((nq, k), -1, np.int64)
        d2 = np.full((nq, k), np.inf, np.float32)
        cnt = np.zeros(nq, np.uint32)
        self.L.oracle_knn_bruteforce(_ptr(xyz, _f32p), len(xyz), _ptr(q, _f32p), nq, k, eps,
                                     _ptr(idx, _i64p), _ptr(d2, _f32p), _ptr(cnt, _u32p))
        return idx, d2, cnt

    def radius_count_bruteforce(self, xyz, queries, r, radii=None):
        xyz = _f32(xyz)
        q = _f32(queries)
        radii = _f32(radii)
        nq = len(xyz) if q is None else len(q)
        cnt = np.zeros(nq, np.uint32)
        self.L.oracle_radius_count_bruteforce(_ptr(xyz, _f32p), len(xyz), _ptr(q, _f32p), nq,
                                              _ptr(radii, _f32p), np.float32(r),
                                              _ptr(cnt, _u32p))
        return cnt


class OracleCloud:
    def __init__(self, oracle, xyz, bbox, node_capacity, max_depth):
        self.o = oracle
        self.L = oracle.L
        self.xyz = _f32(xyz).reshape(-1, 3)
        self.n = len(self.xyz)
        bb = _f32(bbox)
        self.h = self.L.oracle_cloud_create(_ptr(self.xyz, _f32p), self.n, _ptr(bb, _f32p),
                                            node_capacity, max_depth)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.oracle_cloud_destroy(self.h)
            self.h = None

    def size(self):
        return self.L.oracle_cloud_size(self.h)

    def bbox(self):
        out = np.zeros(6, np.float32)
        self.L.oracle_cloud_bbox(self.h, _ptr(out, _f32p))
        return out

    def _nq(self, q):
        return self.n if q is None else len(q)

    def knn(self, queries, k, eps=1e-5, nthreads=None):
        q = _f32(queries)
        nq = self._nq(q)
        idx = np.full((nq, k), -1, np.int64)
        d2 = np.full((nq, k), np.inf, np.float32)
        cnt = np.zeros(nq, np.uint32)
        self.L.oracle_knn(self.h, _ptr(q, _f32p), nq, k, eps, _ptr(idx, _i64p), _ptr(d2, _f32p),
                          _ptr(cnt, _u32p), nthreads or nthreads_default())
        return idx, d2, cnt

    def normals(self, queries, k, eps=1e-5, nthreads=None):
        q = _f32(queries)
        nq = self._nq(q)
        nrm = np.zeros((nq, 3), np.float32)
        gap = np.zeros(nq, np.float32)
        self.L.oracle_estimate_normals(self.h, _ptr(q, _f32p), nq, k, eps, _ptr(nrm, _f32p),
                                       _ptr(gap, _f32p), nthreads or nthreads_default())
        return nrm, gap

    def radius_count(self, queries, r, radii=None, exact_prune=0, nthreads=None):
        q = _f32(queries)
        radii = _f32(radii)
        nq = self._nq(q)
        cnt = np.zeros(nq, np.uint32)
        self.L.oracle_radius(self.h, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                             exact_prune, _ptr(cnt, _u32p), None, None,
                             nthreads or nthreads_default())
        return cnt

    def radius_search(self, queries, r, radii=None, exact_prune=0, nthreads=None):
        q = _f32(queries)
        radii = _f32(radii)
        nq = self._nq(q)
        cnt = self.radius_count(queries, r, radii, exact_prune, nthreads)
        off = np.zeros(nq + 1, np.uint64)
        np.cumsum(cnt, out=off[1:])
        idx = np.zeros(int(off[-1]), np.int64)
        self.L.oracle_radius(self.h, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                             exact_prune, None, _ptr(off, _u64p), _ptr(idx, _i64p),
                             nthreads or nthreads_default())
        return off, idx

    def mean_knn_distance(self, k, eps=1e-5, nthreads=None):
        means = np.zeros(self.n, np.float32)
        mu = self.L.oracle_average_distance_to_neighbors(self.h, k, eps, _ptr(means, _f32p),
                                                         nthreads or nthreads_default())
        return means, np.float32(mu)

    def density_filter(self, radius, threshold, nthreads=None):
        keep = np.zeros(self.n, np.uint8)
        cnt = np.zeros(self.n, np.uint32)
        kept = self.L.oracle_density_filter(self.h, np.float32(radius), threshold,
                                            _ptr(keep, _u8p), _ptr(cnt, _u32p),
                                            nthreads or nthreads_default())
        return keep, cnt, kept


def have_ref():
    return os.path.exists(REF_SO)


def have_ref_smoothing():
    return os.path.exists(REF_SMOOTHING_SO)


class RefSmoothing:
    """The reference's own bilateral_filter_points and WLOP bodies (unmodified headers)."""

    def __init__(self):
        build_oracle()
        L = C.CDLL(REF_SMOOTHING_SO)
        _sz, _dbl = C.c_size_t, C.c_double
        L.ref_bilateral_filter_points.argtypes = [_f32p, _f32p, _sz, _dbl, _dbl, _sz, _f32p]
        L.ref_wlop.argtypes = [_f32p, _sz, _u32p, _sz, _dbl, _dbl, _sz, C.c_int, _f32p]
        self.L = L

    def bilateral_filter_points(self, xyz, normals, sigmaf, sigmag, iterations):
        xyz, normals = _f32(xyz).reshape(-1, 3), _f32(normals).reshape(-1, 3)
        out = np.zeros_like(xyz)
        self.L.ref_bilateral_filter_points(_ptr(xyz, _f32p), _ptr(normals, _f32p), len(xyz),
                                           sigmaf, sigmag, iterations, _ptr(out, _f32p))
        return out

    def wlop(self, xyz, initial, mu, h, iterations, uniform=True):
        xyz = _f32(xyz).reshape(-1, 3)
        initial = np.ascontiguousarray(initial, dtype=np.uint32)
        out = np.zeros((len(initial), 3), np.float32)
        self.L.ref_wlop(_ptr(xyz, _f32p), len(xyz), _ptr(initial, _u32p), len(initial), mu, h,
                        iterations, 1 if uniform else 0, _ptr(out, _f32p))
        return out


def have_ref_orient():
    return os.path.exists(REF_ORIENT_SO)


class RefOrient:
    """The reference's own propagate_normal_orientations (unmodified headers)."""

    def __init__(self):
        build_oracle()
        L = C.CDLL(REF_ORIENT_SO)
        L.ref_propagate_normal_orientations.argtypes = [_f32p, C.c_size_t, _i64p, C.c_size_t,
                                                        _f32p]
        self.L = L

    def propagate_normal_orientations(self, xyz, k, normals, knn=None):
        """knn = None: the reference's own kd-tree neighbours; else n x k int64 (-1 = none)."""
        xyz = _f32(xyz).reshape(-1, 3)
        if knn is not None:
            knn = np.ascontiguousarray(knn, dtype=np.int64)
            k = knn.shape[1]
        out = _f32(normals).reshape(-1, 3).copy()
        self.L.ref_propagate_normal_orientations(_ptr(xyz, _f32p), len(xyz), _ptr(knn, _i64p), k,
                                                 _ptr(out, _f32p))
        return out


def have_ref_ply():
    return os.path.exists(REF_PLY_SO)


class RefPly:
    """The reference's own PLY writer / reader (unmodified pcp/io/ply.hpp) on byte strings."""

    FORMATS = {"ascii": 0, "binary_little_endian": 1, "binary_big_endian": 2}

    def __init__(self):
        build_oracle()
        L = C.CDLL(REF_PLY_SO)
        L.ref_write_ply.restype = C.c_size_t
        L.ref_write_ply.argtypes = [_f32p, C.c_size_t, _f32p, C.c_size_t, C.c_int, _u8p,
                                    C.c_size_t]
        L.ref_read_ply.argtypes = [_u8p, C.c_size_t, _f32p, C.c_size_t, _f32p, C.c_size_t,
                                   C.POINTER(C.c_size_t)]
        self.L = L

    def write(self, xyz, normals, fmt):
        xyz, normals = _f32(xyz).reshape(-1, 3), _f32(normals).reshape(-1, 3)
        cap = 4096 + 64 * (len(xyz) + len(normals))
        buf = np.zeros(cap, np.uint8)
        size = self.L.ref_write_ply(_ptr(xyz, _f32p), len(xyz), _ptr(normals, _f32p),
                                    len(normals), self.FORMATS[fmt], _ptr(buf, _u8p), cap)
        assert size <= cap
        return buf[:size].tobytes()

    def read(self, data, max_rows=1 << 22):
        b = np.frombuffer(data, np.uint8)
        xyz = np.zeros((max_rows, 3), np.float32)
        nrm = np.zeros((max_rows, 3), np.float32)
        counts = (C.c_size_t * 2)()
        self.L.ref_read_ply(_ptr(b, _u8p), len(b), _ptr(xyz, _f32p), max_rows, _ptr(nrm, _f32p),
                            max_rows, counts)
        return xyz[: counts[0]].copy(), nrm[: counts[1]].copy()


class RefBridge:
    """The reference's own octree / kd-tree (unmodified headers) on flat buffers."""

    def __init__(self):
        build_oracle()
        L = C.CDLL(REF_SO)
        L.ref_cloud_create.restype = C.c_void_p
        L.ref_cloud_create.argtypes = [_f32p, C.c_size_t, C.c_int, _f32p, C.c_uint32,
                                       C.c_uint32, C.c_int]
        L.ref_cloud_destroy.argtypes = [C.c_void_p]
        L.ref_octree_size.restype = C.c_size_t
        L.ref_octree_size.argtypes = [C.c_void_p]
        L.ref_octree_bbox.argtypes = [C.c_void_p, _f32p]
        L.ref_knn.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_size_t, C.c_size_t, C.c_double,
                              _i64p, _u32p, C.c_int]
        L.ref_knn_tie_aware.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_size_t, C.c_size_t,
                                        C.c_double, _i64p, _f32p, _u32p, C.c_int]
        L.ref_radius.argtypes = [C.c_void_p, C.c_int, _f32p, C.c_size_t, _f32p, C.c_float,
                                 _u32p, _u64p, _i64p, C.c_int]
        L.ref_average_distance_to_neighbors.restype = C.c_float
        L.ref_average_distance_to_neighbors.argtypes = [C.c_void_p, C.c_int, C.c_size_t, _f32p]
        L.ref_estimate_normals_sample.argtypes = [C.c_void_p, C.c_int, _u32p, C.c_size_t,
                                                  C.c_size_t, _f32p, C.c_int]
        self.L = L

    def cloud(self, xyz, which=2, bbox=None, node_capacity=0, max_depth=0, kd_adaptive=1):
        return RefCloud(self, xyz, which, bbox, node_capacity, max_depth, kd_adaptive)


class RefCloud:
    OCTREE, KDTREE = 0, 1

    def __init__(self, ref, xyz, which, bbox, node_capacity, max_depth, kd_adaptive):
        self.L = ref.L
        self.xyz = _f32(xyz).reshape(-1, 3)
        self.n = len(self.xyz)
        bb = _f32(bbox)
        self.h = self.L.ref_cloud_create(_ptr(self.xyz, _f32p), self.n, which, _ptr(bb, _f32p),
                                         node_capacity, max_depth, kd_adaptive)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ref_cloud_destroy(self.h)
            self.h = None

    def octree_size(self):
        return self.L.ref_octree_size(self.h)

    def octree_bbox(self):
        out = np.zeros(6, np.float32)
        self.L.ref_octree_bbox(self.h, _ptr(out, _f32p))
        return out

    def knn_raw(self, tree, queries, k, eps=1e-5, nthreads=None):
        q = _f32(queries)
        nq = self.n if q is None else len(q)
        idx = np.full((nq, k), -1, np.int64)
        cnt = np.zeros(nq, np.uint32)
        self.L.ref_knn(self.h, tree, _ptr(q, _f32p), nq, k, eps, _ptr(idx, _i64p),
                       _ptr(cnt, _u32p), nthreads or nthreads_default())
        return idx, cnt

    def knn(self, tree, queries, k, eps=1e-5, nthreads=None):
        q = _f32(queries)
        nq = self.n if q is None else len(q)
        idx = np.full((nq, k), -1, np.int64)
        d2 = np.full((nq, k), np.inf, np.float32)
        cnt = np.zeros(nq, np.uint32)
        self.L.ref_knn_tie_aware(self.h, tree, _ptr(q, _f32p), nq, k, eps, _ptr(idx, _i64p),
                                 _ptr(d2, _f32p), _ptr(cnt, _u32p),
                                 nthreads or nthreads_default())
        return idx, d2, cnt

    def radius_count(self, tree, queries, r, radii=None, nthreads=None):
        q = _f32(queries)
        radii = _f32(radii)
        nq = self.n if q is None else len(q)
        cnt = np.zeros(nq, np.uint32)
        self.L.ref_radius(self.h, tree, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                          _ptr(cnt, _u32p), None, None, nthreads or nthreads_default())
        return cnt

    def radius_search(self, tree, queries, r, radii=None, nthreads=None):
        q = _f32(queries)
        radii = _f32(radii)
        nq = self.n if q is None else len(q)
        cnt = self.radius_count(tree, queries, r, radii, nthreads)
        off = np.zeros(nq + 1, np.uint64)
        np.cumsum(cnt, out=off[1:])
        idx = np.zeros(int(off[-1]), np.int64)
        self.L.ref_radius(self.h, tree, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                          None, _ptr(off, _u64p), _ptr(idx, _i64p),
                          nthreads or nthreads_default())
        return off, idx

    def mean_knn_distance(self, tree, k):
        means = np.zeros(self.n, np.float32)
        mu = self.L.ref_average_distance_to_neighbors(self.h, tree, k, _ptr(means, _f32p))
        return means, np.float32(mu)

    def normals_sample(self, tree, sample, k, nthreads=None):
        """estimate_normals' per-element body for the cloud points listed in `sample`"""
        sample = np.ascontiguousarray(sample, dtype=np.uint32)
        out = np.zeros((len(sample), 3), np.float32)
        self.L.ref_estimate_normals_sample(self.h, tree, _ptr(sample, _u32p), len(sample), k,
                                           _ptr(out, _f32p), nthreads or nthreads_default())
        return out
