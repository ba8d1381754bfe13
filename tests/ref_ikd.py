"""ctypes wrapper over oracle/_ref/libref_ikd.so -- the REFERENCE's own ikd-Tree (include/ikd-Tree/ikd_Tree.{h,cpp}) compiled
unmodified from an ImMesh checkout by oracle/Makefile.ref.  tools/make_golden.py drives it to produce the fixtures under
tests/golden/; the tests compare against those fixtures and need neither the library nor the checkout.  `same_knn` is the
kNN comparison they use."""
import ctypes as C
import os
import subprocess

import numpy as np

_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(_ROOT, "oracle", "_ref", "libref_ikd.so")
_lib = None


def build(ref_dir):
    """Compile oracle/_ref/libref_ikd.so from the ImMesh checkout at ref_dir."""
    subprocess.check_call(["make", "-s", "-C", os.path.join(_ROOT, "oracle"), "-f", "Makefile.ref", f"REF={os.path.abspath(ref_dir)}"])
    return _SO


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError("oracle/_ref/libref_ikd.so is not built (ref_ikd.build)")
        L = C.CDLL(_SO)
        L.ref_ikd_create.restype = C.c_void_p
        L.ref_ikd_destroy.argtypes = [C.c_void_p]
        L.ref_ikd_add.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int64]
        L.ref_ikd_knn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
        L.ref_ikd_size.argtypes = [C.c_void_p]
        _lib = L
    return _lib


class RefIkdTree:
    """KD_TREE<ikdTree_PointType> driven like Global_map does: Add_Point one vertex at a time, Nearest_Search."""

    def __init__(self):
        self.L = lib()
        self.h = C.c_void_p(self.L.ref_ikd_create())
        self.n = 0

    def __del__(self):
        try:
            self.L.ref_ikd_destroy(self.h)
        except Exception:
            pass

    def add(self, xyz):
        a = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        self.L.ref_ikd_add(self.h, a.ctypes.data_as(C.c_void_p), a.shape[0], self.n)
        self.n += a.shape[0]

    def knn(self, q, k, max_dist=float("inf")):
        a = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, 3)
        idx = np.zeros((a.shape[0], k), dtype=np.int64)
        d2 = np.zeros((a.shape[0], k), dtype=np.float32)
        cnt = np.zeros(a.shape[0], dtype=np.int32)
        self.L.ref_ikd_knn(self.h, a.ctypes.data_as(C.c_void_p), a.shape[0], k, max_dist, idx.ctypes.data_as(C.c_void_p),
                           d2.ctypes.data_as(C.c_void_p), cnt.ctypes.data_as(C.c_void_p))
        return idx, d2, cnt


def same_knn(idx_a, d2_a, idx_b, d2_b):
    """kNN equality up to the order inside groups of EXACTLY equal float distances (tie order in the ikd-Tree depends on the
    tree shape, ikd_Tree.cpp:1123; ours is defined as lower id first)."""
    if not np.array_equal(d2_a, d2_b):
        return False
    for r in range(idx_a.shape[0]):
        if np.array_equal(idx_a[r], idx_b[r]):
            continue
        d = d2_a[r]
        for v in np.unique(d):
            m = d == v
            if sorted(idx_a[r][m].tolist()) != sorted(idx_b[r][m].tolist()):
                return False
    return True
