"""ctypes loader for tests/emu/libpcpx_emu_box.so — the emulated index of tests/emu/emu.cu plus
the box traversal (box_visit, box_core.cuh) run on the host.

TEST HARNESS ONLY: lets the CPU-only suite check the box search against a brute force. It is not
a fallback of the product; libpcpx.so contains none of it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_lib import CSRC, EMU_DIR, ROOT, _f32, _f32p, _ptr, _u32p, _u64p

BOX_SRC = os.path.join(EMU_DIR, "emu_box.cu")
BOX_SO = os.path.join(EMU_DIR, "libpcpx_emu_box.so")


def build_box_emu(force=False):
    srcs = [BOX_SRC, os.path.join(EMU_DIR, "emu.cu")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp"))
    ]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(BOX_SO) or os.path.getmtime(BOX_SO) < newest:
        subprocess.run(
            ["nvcc", "-std=c++17", "-O2", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013",
             "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
             "-I", os.path.join(ROOT, "include"), "-I", CSRC, BOX_SRC, "-o", BOX_SO],
            check=True, capture_output=True)


class BoxEmu:
    def __init__(self):
        build_box_emu()
        L = C.CDLL(BOX_SO)
        L.emu_index_create.restype = C.c_void_p
        L.emu_index_create.argtypes = [_f32p, C.c_size_t, C.c_int, _f32p, C.c_uint32, C.c_uint32]
        L.emu_index_destroy.argtypes = [C.c_void_p]
        L.emu_index_info.argtypes = [C.c_void_p, _u64p, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                     _u64p]
        L.emu_box_search.argtypes = [C.c_void_p, _f32p, C.c_size_t, C.c_size_t, _f32p, _u32p,
                                     _u64p, _u32p, _u64p]
        self.L = L

    def index(self, xyz, voxel_grid=None, max_level=0):
        return BoxEmuIndex(self.L, xyz, voxel_grid, max_level)


class BoxEmuIndex:
    def __init__(self, L, xyz, voxel_grid, max_level):
        self.L = L
        self.xyz = _f32(xyz).reshape(-1, 3)
        self.n = len(self.xyz)
        self.voxel = None if voxel_grid is None else _f32(np.concatenate(voxel_grid))
        self.h = L.emu_index_create(_ptr(self.xyz, _f32p), self.n, 0 if self.voxel is None else 1,
                                    _ptr(self.voxel, _f32p), max_level, 0)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.emu_index_destroy(self.h)
            self.h = None

    def info(self):
        n, slots = C.c_uint64(), C.c_uint64()
        lcap, lfine = C.c_int(), C.c_int()
        self.L.emu_index_info(self.h, C.byref(n), C.byref(lcap), C.byref(lfine), C.byref(slots))
        return dict(n_indexed=n.value, lcap=lcap.value, lfine=lfine.value)

    def box_search(self, boxes):
        """(offsets, idx, spans): CSR lists in the device fill's order, and the number of INSIDE
        spans of every box."""
        b = _f32(boxes).reshape(-1, 6)
        nb = len(b)
        cnt = np.zeros(nb, np.uint32)
        spans = np.zeros(nb, np.uint64)
        self.L.emu_box_search(self.h, _ptr(b, _f32p), nb, 6, _ptr(self.voxel, _f32p),
                              _ptr(cnt, _u32p), None, None, _ptr(spans, _u64p))
        off = np.zeros(nb + 1, np.uint64)
        off[1:] = np.cumsum(cnt, dtype=np.uint64)
        idx = np.zeros(max(int(off[-1]), 1), np.uint32)
        cnt2 = np.zeros(nb, np.uint32)
        self.L.emu_box_search(self.h, _ptr(b, _f32p), nb, 6, _ptr(self.voxel, _f32p),
                              _ptr(cnt2, _u32p), _ptr(off, _u64p), _ptr(idx, _u32p), None)
        assert np.array_equal(cnt, cnt2)
        return off, idx[:int(off[-1])], spans


def bruteforce_boxes(xyz, boxes, indexed=None):
    """The fp32 predicate min <= p <= max on every axis, box by box: a list of ascending original
    indices per box.  `indexed`: mask of the points the index holds (a voxel grid's)."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    boxes = np.asarray(boxes, np.float32).reshape(-1, 6)
    keep = np.ones(len(xyz), bool) if indexed is None else np.asarray(indexed, bool)
    out = []
    for b in boxes:
        m = keep & np.all((xyz >= b[:3]) & (xyz <= b[3:]), axis=1)
        out.append(np.nonzero(m)[0].astype(np.uint32))
    return out


def split_csr(off, idx):
    return [idx[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]
