"""ctypes binding of include/pcpx.h.  Buffers may be numpy arrays (host) or torch CUDA tensors
(device pointers are passed straight through; results can stay resident in HBM)."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCPX_LIB", os.path.join(HERE, "lib", "libpcpx.so"))  # PCPX_LIB: experimental builds
if os.environ.get("PCPX_LIB"):  # an experimental build next to the product (build.py --out=...)
    LIB_PATH = os.environ["PCPX_LIB"]
NO_NEIGHBOUR = 0xFFFFFFFF
NOISE = 0xFFFFFFFF  # PCPX_NOISE: the label of a point in no cluster


class PcpxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("pcpx error %d: %s" % (code, msg))
        self.code = code


class IndexParams(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("use_voxel_grid", C.c_int32),
        ("voxel_min", C.c_float * 3),
        ("voxel_max", C.c_float * 3),
        ("max_level", C.c_uint32),
        ("min_cell_occupancy", C.c_uint32),
        ("n_devices", C.c_uint32),
        ("devices", C.c_int32 * 8),
        ("shard_mode", C.c_uint32),
        ("reserved", C.c_uint32 * 6),
    ]


class IndexInfo(C.Structure):
    _fields_ = [
        ("n_input", C.c_uint64),
        ("n_indexed", C.c_uint64),
        ("bbox_min", C.c_float * 3),
        ("bbox_max", C.c_float * 3),
        ("code_bits", C.c_uint32),
        ("finest_level", C.c_uint32),
        ("n_cells", C.c_uint64),
        ("device_bytes", C.c_uint64),
        ("device", C.c_int32),
        ("build_ms", C.c_float),
        ("n_devices", C.c_uint32),
    ]


class Timings(C.Structure):
    _fields_ = [
        ("build_ms", C.c_float),
        ("sort_ms", C.c_float),
        ("query_sort_ms", C.c_float),
        ("kernel_ms", C.c_float),
        ("total_ms", C.c_float),
        ("kernel_launches", C.c_uint32),
        ("retry_queries", C.c_uint32),
        ("deferred_queries", C.c_uint32),
        ("expanded_queries", C.c_uint32),
    ]


class IcpParams(C.Structure):
    _fields_ = [
        ("metric", C.c_uint32),
        ("max_iterations", C.c_uint32),
        ("max_distance", C.c_float),
        ("rotation_tolerance", C.c_double),
        ("translation_tolerance", C.c_double),
        ("reserved", C.c_uint32 * 8),
    ]


class IcpResult(C.Structure):
    _fields_ = [
        ("iterations", C.c_uint32),
        ("stop_reason", C.c_uint32),
        ("n_correspondences", C.c_uint64),
        ("fitness", C.c_double),
        ("rmse", C.c_double),
    ]


ICP_METRICS = {"point_to_plane": 0, "point_to_point": 1}
ICP_STOP = {0: "converged", 1: "max_iterations", 2: "too_few"}


_SIGNATURES = {
    # name: (restype, argtypes)
    "pcpx_device_count": (C.c_int, []),
    "pcpx_last_error": (C.c_char_p, []),
    "pcpx_index_create": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.POINTER(IndexParams),
                                    C.POINTER(C.c_void_p)]),
    "pcpx_index_destroy": (None, [C.c_void_p]),
    "pcpx_index_info_get": (C.c_int, [C.c_void_p, C.POINTER(IndexInfo)]),
    "pcpx_index_bbox": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "pcpx_knn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_uint32,
                           C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcpx_radius_count": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                    C.c_float, C.c_void_p]),
    "pcpx_radius_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                     C.c_float, C.c_void_p, C.POINTER(C.c_void_p), C.c_int]),
    "pcpx_box_count": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p]),
    "pcpx_box_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                  C.POINTER(C.c_void_p), C.c_int]),
    "pcpx_free": (None, [C.c_void_p, C.c_int]),
    "pcpx_estimate_normals": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                        C.c_uint32, C.c_double, C.c_void_p]),
    "pcpx_estimate_tangent_planes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                               C.c_uint32, C.c_double, C.c_void_p, C.c_void_p]),
    "pcpx_estimate_normals_radius": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                               C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "pcpx_estimate_tangent_planes_radius": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t,
                                                      C.c_size_t, C.c_void_p, C.c_float,
                                                      C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcpx_normals_from_neighbourhoods": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int,
                                                   C.c_void_p]),
    "pcpx_mean_knn_distance": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.c_void_p,
                                         C.POINTER(C.c_double)]),
    "pcpx_density_filter": (C.c_int, [C.c_void_p, C.c_float, C.c_uint32, C.c_void_p, C.c_void_p,
                                      C.POINTER(C.c_size_t)]),
    "pcpx_cluster_by_density": (C.c_int, [C.c_void_p, C.c_float, C.c_uint32, C.c_void_p,
                                          C.POINTER(C.c_uint64)]),
    "pcpx_nearest_within": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_size_t,
                                      C.c_void_p, C.c_float, C.c_void_p, C.c_void_p]),
    "pcpx_icp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t,
                           C.POINTER(IcpParams), C.c_void_p, C.c_void_p, C.POINTER(IcpResult),
                           C.c_void_p]),
    "pcpx_bilateral_filter_points": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                               C.c_size_t, C.c_double, C.c_double, C.c_uint32,
                                               C.c_int, C.c_void_p, C.POINTER(C.c_float)]),
    "pcpx_bilateral_filter_normals": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                                C.c_size_t, C.c_double, C.c_double, C.c_uint32,
                                                C.c_int, C.c_void_p, C.POINTER(C.c_float)]),
    "pcpx_wlop": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t,
                            C.c_double, C.c_double, C.c_uint32, C.c_int, C.c_uint32, C.c_int,
                            C.c_void_p, C.POINTER(C.c_float)]),
    "pcpx_orient_normals": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.c_int, C.c_void_p,
                                      C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "pcpx_orient_normals_graph": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p,
                                            C.c_uint32, C.c_int, C.c_int, C.c_void_p,
                                            C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
    "pcpx_extract_bands": (C.c_int, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int, C.c_float,
                                     C.c_float, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p,
                                     C.c_void_p]),
    "pcpx_last_timings": (C.c_int, [C.c_void_p, C.POINTER(Timings)]),
    "pcpx_set_tuning": (C.c_int, [C.c_char_p, C.c_double]),
    "pcpx_trim": (C.c_int, [C.c_int]),
    "pcpx_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "pcpx_host_free": (None, [C.c_void_p]),
    "pcpx_debug_knn_stats": (C.c_int, [C.c_void_p, C.c_uint32, C.c_double, C.c_void_p]),
}

_lib = None


def exported_symbols():
    """Names include/pcpx.h declares; the CPU suite checks the library exports each of them."""
    return sorted(_SIGNATURES)


def lib():
    """The loaded libpcpx.so.  Fails loudly when it has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PcpxError(-3, "libpcpx.so is not built (%s); run `python "
                            "point-cloud-processing_b200/build.py` — there is no CPU fallback"
                            % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            f = getattr(L, name)  # AttributeError = a declared symbol is missing
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _check(rc):
    if rc != 0:
        raise PcpxError(rc, lib().pcpx_last_error().decode("utf-8", "replace"))


def device_count():
    return lib().pcpx_device_count()


def trim(device=0):
    """free the library's cache of device blocks on `device` (after the device went idle)"""
    _check(lib().pcpx_trim(int(device)))


def set_tuning(name, value):
    _check(lib().pcpx_set_tuning(name.encode(), float(value)))


def normals_from_neighbourhoods(nbr_xyz, offsets, device=-1):
    """PCA normal of caller-supplied neighbourhoods (CSR over packed xyz)."""
    nbr = np.ascontiguousarray(nbr_xyz, np.float32).reshape(-1, 3)
    off = np.ascontiguousarray(offsets, np.uint64)
    n = len(off) - 1
    out = np.zeros((n, 3), np.float32)
    _check(lib().pcpx_normals_from_neighbourhoods(nbr.ctypes.data, off.ctypes.data, n, device,
                                                  out.ctypes.data))
    return out


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _out_rows(like, n, out):
    """result buffer of n xyz rows: `out` if given, else same kind (numpy / torch) as `like`"""
    if out is not None:
        return out
    if _is_torch(like):
        import torch
        return torch.empty((n, 3), dtype=torch.float32, device=like.device)
    return np.zeros((n, 3), np.float32)


def _out_vec(like, n, dtype):
    """result vector of n entries of the same kind (numpy / torch) as `like`"""
    if _is_torch(like):
        import torch
        tdt = {np.dtype(np.uint32): torch.int32, np.dtype(np.float32): torch.float32}
        return torch.empty(n, dtype=tdt[np.dtype(dtype)], device=like.device)
    return np.zeros(n, dtype)


def _bilateral(fn, xyz, normals, sigmaf, sigmag, iterations, device, out):
    n = _count(xyz)
    bx, bn = _Buf(xyz, np.float32), _Buf(normals, np.float32)
    res = _out_rows(xyz, n, out)
    bo = _Buf(res, np.float32, writable=True)
    ms = C.c_float(-1.0)
    _check(fn(bx.ptr, n, 12, bn.ptr, 12, float(sigmaf), float(sigmag), int(iterations), device,
              bo.ptr, C.byref(ms)))
    return res, ms.value


def bilateral_filter_points(xyz, normals, sigmaf, sigmag, iterations=1, device=-1, out=None,
                            want_ms=False):
    """pcp::algorithm::bilateral_filter_points on the GPU (include/pcpx.h)."""
    res, ms = _bilateral(lib().pcpx_bilateral_filter_points, xyz, normals, sigmaf, sigmag,
                         iterations, device, out)
    return (res, ms) if want_ms else res


def bilateral_filter_normals(xyz, normals, sigmaf, sigmag, iterations=1, device=-1, out=None,
                             want_ms=False):
    """pcp::algorithm::bilateral_filter_normals on the GPU (include/pcpx.h)."""
    res, ms = _bilateral(lib().pcpx_bilateral_filter_normals, xyz, normals, sigmaf, sigmag,
                         iterations, device, out)
    return (res, ms) if want_ms else res


def orient_normals_graph(xyz, neighbours, normals, nearest_first=False, device=-1):
    """propagate_normal_orientations over an explicit directed graph: `neighbours` is n x k
    uint32 (NO_NEIGHBOUR = unused slot); `normals` is updated in place and returned."""
    n = _count(xyz)
    bx = _Buf(xyz, np.float32)
    if not _is_torch(neighbours):
        neighbours = np.ascontiguousarray(neighbours, np.uint32)
    k = neighbours.shape[1]
    bn = _Buf(neighbours)
    if not _is_torch(normals):
        assert normals.dtype == np.float32 and normals.flags["C_CONTIGUOUS"]
    bo = _Buf(normals, np.float32, True)
    _check(lib().pcpx_orient_normals_graph(bx.ptr, n, 12, bn.ptr, k, 1 if nearest_first else 0,
                                           device, bo.ptr, None, None))
    return normals


def extract_bands(xyz, axis, below, above, out_below, out_above, counts, stream=None):
    """Boundary strips of a device-resident slab (CUDA tensors throughout; see pcpx.h).
    `counts`: a 2-element int64 CUDA tensor or numpy uint64 array."""
    n = _count(xyz)
    cap = min(out_below.shape[0], out_above.shape[0])
    cptr = counts.data_ptr() if _is_torch(counts) else counts.ctypes.data
    _check(lib().pcpx_extract_bands(xyz.data_ptr(), n, 12, int(axis), float(below), float(above),
                                    out_below.data_ptr(), out_above.data_ptr(), cap, cptr,
                                    stream))


def wlop(xyz, n_out, h, mu=0.45, iterations=10, uniform=True, initial=None, seed=0, device=-1,
         out=None, want_ms=False):
    """pcp::algorithm::wlop::wlop on the GPU; `initial` = the start set's indices into xyz."""
    n = _count(xyz)
    bx = _Buf(xyz, np.float32)
    bi = _Buf(initial, np.uint32 if not _is_torch(initial) else None)
    if initial is not None:
        n_out = initial.numel() if _is_torch(initial) else len(bi.obj)
    res = _out_rows(xyz, n_out, out)
    bo = _Buf(res, np.float32, writable=True)
    ms = C.c_float(-1.0)
    _check(lib().pcpx_wlop(bx.ptr, n, 12, bi.ptr, int(n_out), float(mu), float(h),
                           int(iterations), 1 if uniform else 0, int(seed), device, bo.ptr,
                           C.byref(ms)))
    return (res, ms.value) if want_ms else res


class _Buf:
    """pointer + keep-alive for a numpy array / torch tensor / None"""

    def __init__(self, x, dtype=None, writable=False):
        self.obj = x
        if x is None:
            self.ptr = None
        elif _is_torch(x):
            assert x.is_contiguous()
            self.ptr = x.data_ptr()
        else:
            if not writable:
                x = np.ascontiguousarray(x, dtype=dtype)
                self.obj = x
            assert x.flags["C_CONTIGUOUS"]
            if dtype is not None:
                assert x.dtype == np.dtype(dtype), (x.dtype, dtype)
            self.ptr = x.ctypes.data


def _count(x):
    if x is None:
        return 0
    if _is_torch(x):
        return x.shape[0] if x.dim() == 2 else x.numel() // 3
    x = np.asarray(x)
    return x.shape[0] if x.ndim == 2 else x.size // 3


def _count_boxes(x):
    if _is_torch(x):
        return x.numel() // 6
    return np.asarray(x).size // 6


class Index:
    """GPU-resident spatial index over a cloud (include/pcpx.h: pcpx_index_create)."""

    def __init__(self, xyz, device=-1, voxel_grid=None, max_level=0, min_cell_occupancy=0,
                 stride_bytes=12, devices=None):
        """devices: list of CUDA ordinals — the index is replicated on all of them and kNN-shaped
        calls are sharded over them (pcpx_index_params.devices); devices[0] is the primary."""
        self._h = None
        n = _count(xyz)
        buf = _Buf(xyz, np.float32)
        prm = IndexParams()
        prm.device = device
        if devices:
            if len(devices) > 8:
                raise PcpxError(-1, "at most 8 devices behind one handle")
            prm.n_devices = len(devices)
            for i, d in enumerate(devices):
                prm.devices[i] = int(d)
        if voxel_grid is not None:
            prm.use_voxel_grid = 1
            lo, hi = voxel_grid
            for a in range(3):
                prm.voxel_min[a] = float(lo[a])
                prm.voxel_max[a] = float(hi[a])
        prm.max_level = max_level
        prm.min_cell_occupancy = min_cell_occupancy
        h = C.c_void_p()
        _check(lib().pcpx_index_create(buf.ptr, n, stride_bytes, C.byref(prm), C.byref(h)))
        self._h = h
        self.n = n

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.pcpx_index_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- facts ---------------------------------------------------------------------------
    def info(self):
        i = IndexInfo()
        _check(lib().pcpx_index_info_get(self._h, C.byref(i)))
        return dict(n_input=i.n_input, n_indexed=i.n_indexed,
                    bbox_min=np.array(i.bbox_min[:], np.float32),
                    bbox_max=np.array(i.bbox_max[:], np.float32), code_bits=i.code_bits,
                    finest_level=i.finest_level, n_cells=i.n_cells,
                    device_bytes=i.device_bytes, device=i.device, build_ms=i.build_ms,
                    n_devices=i.n_devices)

    def bbox(self):
        lo, hi = (C.c_float * 3)(), (C.c_float * 3)()
        _check(lib().pcpx_index_bbox(self._h, lo, hi))
        return np.array(lo[:], np.float32), np.array(hi[:], np.float32)

    def timings(self):
        t = Timings()
        _check(lib().pcpx_last_timings(self._h, C.byref(t)))
        return {f: getattr(t, f) for f, _ in Timings._fields_}

    def knn_stats(self, k, eps=1e-5):
        out = np.zeros(4, np.uint64)
        _check(lib().pcpx_debug_knn_stats(self._h, k, eps, out.ctypes.data))
        return out

    # ---- queries -------------------------------------------------------------------------
    def _nq(self, queries):
        return self.n if queries is None else _count(queries)

    def knn(self, queries, k, eps=1e-5, out_idx=None, out_d2=None, out_count=None,
            want_d2=True, want_count=True):
        """Rows of ``k`` original indices nearest -> furthest (pad NO_NEIGHBOUR)."""
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        if out_idx is None:
            out_idx = np.full((nq, k), NO_NEIGHBOUR, np.uint32)
        if out_d2 is None and want_d2:
            out_d2 = np.full((nq, k), np.inf, np.float32)
        if out_count is None and want_count:
            out_count = np.zeros(nq, np.uint32)
        bi, bd, bc = (_Buf(out_idx, np.uint32, True), _Buf(out_d2, np.float32, True),
                      _Buf(out_count, np.uint32, True))
        _check(lib().pcpx_knn(self._h, q.ptr, nq, 12, k, eps, bi.ptr, bd.ptr, bc.ptr))
        return out_idx, out_d2, out_count

    def radius_count(self, queries, radius, radii=None, out_count=None):
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        r = _Buf(radii, np.float32)
        if out_count is None:
            out_count = np.zeros(nq, np.uint32)
        bc = _Buf(out_count, np.uint32, True)
        _check(lib().pcpx_radius_count(self._h, q.ptr, nq, 12, r.ptr, float(radius), bc.ptr))
        return out_count

    def radius_search(self, queries, radius, radii=None, sorted=False):
        """CSR (offsets[nq + 1], indices) — host arrays; sorted: every list ascending by index
        (PCPX_RADIUS_SORTED), otherwise traversal order."""
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        r = _Buf(radii, np.float32)
        off = np.zeros(nq + 1, np.uint64)
        p = C.c_void_p()
        _check(lib().pcpx_radius_search(self._h, q.ptr, nq, 12, r.ptr, float(radius),
                                        off.ctypes.data, C.byref(p), 2 if sorted else 0))
        total = int(off[-1])
        try:
            idx = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)),
                                        shape=(max(total, 1),))[:total].copy()
        finally:
            lib().pcpx_free(p, 0)
        return off, idx

    def box_count(self, boxes, out_count=None):
        """Size of every box's result; `boxes` is (nb, 6) {min xyz, max xyz}, a numpy array or a
        CUDA tensor (then the counts are a CUDA tensor too, unless out_count is given)."""
        nb = _count_boxes(boxes)
        b = _Buf(boxes, np.float32)
        if out_count is None:
            if _is_torch(boxes):
                import torch
                out_count = torch.empty(nb, dtype=torch.int32, device=boxes.device)
            else:
                out_count = np.zeros(nb, np.uint32)
        bc = _Buf(out_count, np.uint32, True)
        _check(lib().pcpx_box_count(self._h, b.ptr, nb, 24, bc.ptr))
        return out_count

    def box_search(self, boxes, sorted=False):
        """CSR (offsets[nb + 1], indices) of the indexed points inside every box — host arrays;
        sorted: every list ascending by index (PCPX_RADIUS_SORTED), otherwise traversal order."""
        nb = _count_boxes(boxes)
        b = _Buf(boxes, np.float32)
        off = np.zeros(nb + 1, np.uint64)
        p = C.c_void_p()
        _check(lib().pcpx_box_search(self._h, b.ptr, nb, 24, off.ctypes.data, C.byref(p),
                                     2 if sorted else 0))
        total = int(off[-1])
        try:
            idx = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)),
                                        shape=(max(total, 1),))[:total].copy()
        finally:
            lib().pcpx_free(p, 0)
        return off, idx

    def estimate_normals(self, queries, k, eps=1e-5, out=None):
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        if out is None:
            out = np.zeros((nq, 3), np.float32)
        bo = _Buf(out, np.float32, True)
        _check(lib().pcpx_estimate_normals(self._h, q.ptr, nq, 12, k, eps, bo.ptr))
        return out

    def estimate_tangent_planes(self, queries, k, eps=1e-5):
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        pts = np.zeros((nq, 3), np.float32)
        nrm = np.zeros((nq, 3), np.float32)
        _check(lib().pcpx_estimate_tangent_planes(self._h, q.ptr, nq, 12, k, eps,
                                                  pts.ctypes.data, nrm.ctypes.data))
        return pts, nrm

    def estimate_normals_radius(self, queries, radius, radii=None, out=None, out_count=None):
        """PCA normal of every query's ball (the set radius_search returns); `radii` gives one
        radius per query.  Results are numpy arrays, or CUDA tensors when the queries are;
        out_count, when given, receives the ball sizes."""
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        r = _Buf(radii, np.float32)
        out = _out_rows(queries, nq, out)
        bo, bc = _Buf(out, np.float32, True), _Buf(out_count, np.uint32, True)
        _check(lib().pcpx_estimate_normals_radius(self._h, q.ptr, nq, 12, r.ptr, float(radius),
                                                  bo.ptr, bc.ptr))
        return out

    def estimate_tangent_planes_radius(self, queries, radius, radii=None):
        """(centroids, normals, counts) of every query's ball; an empty ball gives a NaN
        centroid, normal (0,0,1) and count 0."""
        nq = self._nq(queries)
        q = _Buf(queries, np.float32)
        r = _Buf(radii, np.float32)
        pts, nrm = _out_rows(queries, nq, None), _out_rows(queries, nq, None)
        if _is_torch(queries):
            import torch
            cnt = torch.empty(nq, dtype=torch.int32, device=queries.device)
        else:
            cnt = np.zeros(nq, np.uint32)
        bp, bn, bc = _Buf(pts, np.float32, True), _Buf(nrm, np.float32, True), _Buf(cnt)
        _check(lib().pcpx_estimate_tangent_planes_radius(self._h, q.ptr, nq, 12, r.ptr,
                                                         float(radius), bp.ptr, bn.ptr, bc.ptr))
        return pts, nrm, cnt

    def mean_knn_distance(self, k, eps=1e-5):
        per = np.zeros(self.n, np.float32)
        mean = C.c_double()
        _check(lib().pcpx_mean_knn_distance(self._h, k, eps, per.ctypes.data, C.byref(mean)))
        return per, mean.value

    def density_filter(self, radius, threshold, want_points=True, out_mask=None, out_xyz=None):
        if out_mask is None:
            out_mask = np.zeros(self.n, np.uint8)
        if out_xyz is None and want_points:
            out_xyz = np.zeros((self.n, 3), np.float32)
        bm = _Buf(out_mask, np.uint8, True)
        bx = _Buf(out_xyz, np.float32, True)
        kept = C.c_size_t()
        _check(lib().pcpx_density_filter(self._h, float(radius), int(threshold), bm.ptr, bx.ptr,
                                         C.byref(kept)))
        if out_xyz is not None and not _is_torch(out_xyz):
            out_xyz = out_xyz[: kept.value]
        return out_mask, out_xyz, kept.value

    def cluster_by_density(self, radius, min_points, out_labels=None):
        """DBSCAN over the exact ball of radius_search: (labels, n_clusters).  labels[i] is the
        cluster of point i, 0 .. n_clusters - 1 in ascending order of each cluster's smallest core
        index, or NOISE.  out_labels: n entries, a numpy uint32 array or a CUDA
        tensor of 32-bit integers (a new numpy array when None)."""
        if out_labels is None:
            out_labels = np.zeros(self.n, np.uint32)
        bl = _Buf(out_labels, np.uint32, True)
        nc = C.c_uint64()
        _check(lib().pcpx_cluster_by_density(self._h, float(radius), int(min_points), bl.ptr,
                                             C.byref(nc)))
        return out_labels, nc.value

    def nearest_within(self, queries, max_distance, transform=None, out_idx=None, out_d2=None):
        """Bounded nearest neighbour of every query mapped by the 4 x 4 rigid `transform` (None:
        the queries as they are): (idx, d2), NO_NEIGHBOUR and +inf where no indexed point lies
        within max_distance.  Numpy arrays or CUDA tensors (results follow the queries' kind
        unless out_idx / out_d2 are given)."""
        nq = _count(queries)
        q = _Buf(queries, np.float32)
        tf = None if transform is None else np.ascontiguousarray(transform, np.float64).reshape(16)
        if out_idx is None:
            out_idx = _out_vec(queries, nq, np.uint32)
        if out_d2 is None:
            out_d2 = _out_vec(queries, nq, np.float32)
        bi, bd = _Buf(out_idx, np.uint32, True), _Buf(out_d2, np.float32, True)
        _check(lib().pcpx_nearest_within(self._h, q.ptr, nq, 12,
                                         None if tf is None else tf.ctypes.data,
                                         float(max_distance), bi.ptr, bd.ptr))
        return out_idx, out_d2

    def icp(self, source, max_distance, normals=None, metric="point_to_plane", init=None,
            max_iterations=30, rotation_tolerance=0, translation_tolerance=0,
            out_correspondences=None, source_stride_bytes=12, normal_stride_bytes=12):
        """Rigid registration of `source` to the indexed cloud (pcpx_icp): (T, result).  T is the
        4 x 4 float64 transform mapping the source onto the target; result holds iterations,
        stop_reason ("converged", "max_iterations", "too_few"), n_correspondences, fitness and
        rmse.  `normals`: the target's n x 3 normals (point-to-plane).  Numpy arrays or CUDA
        tensors; out_correspondences (ns entries) receives every source point's pair."""
        ns = _count(source) if source_stride_bytes == 12 else (
            (source.numel() if _is_torch(source) else np.asarray(source).size) * 4
            // source_stride_bytes)
        bs, bn = _Buf(source, np.float32), _Buf(normals, np.float32)
        prm = IcpParams()
        prm.metric = ICP_METRICS[metric] if isinstance(metric, str) else int(metric)
        prm.max_iterations = int(max_iterations)
        prm.max_distance = float(max_distance)
        prm.rotation_tolerance = float(rotation_tolerance)
        prm.translation_tolerance = float(translation_tolerance)
        ti = None if init is None else np.ascontiguousarray(init, np.float64).reshape(16)
        T = np.zeros((4, 4), np.float64)
        res = IcpResult()
        bc = _Buf(out_correspondences, np.uint32, True)
        _check(lib().pcpx_icp(self._h, bn.ptr, normal_stride_bytes, bs.ptr, ns, source_stride_bytes,
                              C.byref(prm), None if ti is None else ti.ctypes.data,
                              T.ctypes.data, C.byref(res), bc.ptr))
        return T, dict(iterations=res.iterations,
                       stop_reason=ICP_STOP.get(res.stop_reason, res.stop_reason),
                       n_correspondences=res.n_correspondences, fitness=res.fitness,
                       rmse=res.rmse)

    def orient_normals(self, normals, k, eps=1e-5, nearest_first=False, want_stats=False):
        """propagate_normal_orientations over the kNN graph; `normals` (numpy array or CUDA
        tensor, n x 3 float32) is updated IN PLACE and returned."""
        if not _is_torch(normals):
            assert normals.dtype == np.float32 and normals.flags["C_CONTIGUOUS"]
        b = _Buf(normals, np.float32, True)
        levels, reached = C.c_uint32(), C.c_uint64()
        _check(lib().pcpx_orient_normals(self._h, int(k), float(eps), 1 if nearest_first else 0,
                                         b.ptr, C.byref(levels), C.byref(reached)))
        return (normals, levels.value, reached.value) if want_stats else normals
