"""ctypes loader for tests/emu/libpcpx_emu_ball.so — the emulated index of tests/emu/emu.cu plus
the ball PCA device body (radius_normal, normals_core.cuh) run on the host.

TEST HARNESS ONLY: lets the CPU-only suite check the ball PCA against the oracle. It is not a
fallback of the product; libpcpx.so contains none of it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

from emu_lib import CSRC, EMU_DIR, ROOT, _f32, _f32p, _ptr, _u32p

BALL_SRC = os.path.join(EMU_DIR, "emu_ball.cu")
BALL_SO = os.path.join(EMU_DIR, "libpcpx_emu_ball.so")


def build_ball_emu(force=False):
    srcs = [BALL_SRC, os.path.join(EMU_DIR, "emu.cu")] + [
        os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".hpp"))
    ]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(BALL_SO) or os.path.getmtime(BALL_SO) < newest:
        subprocess.run(
            ["nvcc", "-std=c++17", "-O2", "-Wno-deprecated-gpu-targets", "-diag-suppress", "20013",
             "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared",
             "-I", os.path.join(ROOT, "include"), "-I", CSRC, BALL_SRC, "-o", BALL_SO],
            check=True, capture_output=True)


class BallEmu:
    def __init__(self):
        build_ball_emu()
        L = C.CDLL(BALL_SO)
        L.emu_index_create.restype = C.c_void_p
        L.emu_index_create.argtypes = [_f32p, C.c_size_t, C.c_int, _f32p, C.c_uint32, C.c_uint32]
        L.emu_index_destroy.argtypes = [C.c_void_p]
        L.emu_radius.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_float, _u32p,
                                 C.POINTER(C.c_uint64), _u32p]
        L.emu_radius_normals.argtypes = [C.c_void_p, _f32p, C.c_size_t, _f32p, C.c_float, _f32p,
                                         _f32p, _u32p]
        self.L = L

    def index(self, xyz, bbox=None):
        return BallEmuIndex(self.L, xyz, bbox)


class BallEmuIndex:
    def __init__(self, L, xyz, bbox):
        self.L = L
        self.xyz = _f32(xyz).reshape(-1, 3)
        self.n = len(self.xyz)
        bb = _f32(bbox)
        self.h = L.emu_index_create(_ptr(self.xyz, _f32p), self.n, 0 if bb is None else 1,
                                    _ptr(bb, _f32p), 0, 0)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.emu_index_destroy(self.h)
            self.h = None

    def radius_count(self, queries, r, radii=None):
        q, radii = _f32(queries), _f32(radii)
        nq = self.n if q is None else len(q)
        cnt = np.zeros(nq, np.uint32)
        self.L.emu_radius(self.h, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                          _ptr(cnt, _u32p), None, None)
        return cnt

    def radius_normals(self, queries, r, radii=None):
        """(normals, centroids, counts) of every query's ball, by the device body."""
        q, radii = _f32(queries), _f32(radii)
        nq = self.n if q is None else len(q)
        nrm = np.zeros((nq, 3), np.float32)
        ctr = np.zeros((nq, 3), np.float32)
        cnt = np.zeros(nq, np.uint32)
        self.L.emu_radius_normals(self.h, _ptr(q, _f32p), nq, _ptr(radii, _f32p), np.float32(r),
                                  _ptr(nrm, _f32p), _ptr(ctr, _f32p), _ptr(cnt, _u32p))
        return nrm, ctr, cnt
