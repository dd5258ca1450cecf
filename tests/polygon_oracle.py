"""Loader of tests/polygon_oracle.c, the sequential polygonizer the tests and tools/time_polygonize.py compare
dm_polygonize against.  TEST INFRASTRUCTURE ONLY.  The library is compiled with gcc into a temporary directory once
per process, so the source tree is never written."""
from __future__ import annotations

import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "polygon_oracle.c")

_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        d = tempfile.mkdtemp(prefix="polygon_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libpolygon_oracle.so")
        r = subprocess.run(["gcc", "-O2", "-std=c99", "-shared", "-fPIC", "-o", so, SRC], capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("gcc failed on polygon_oracle.c:\n" + r.stderr)
        L = ctypes.CDLL(so)
        p, i64, i = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
        L.dmo_poly_successor.restype = i
        L.dmo_poly_successor.argtypes = [p, i64, i64, i64, i64, i, p]
        L.dmo_polygonize.restype = i
        L.dmo_polygonize.argtypes = [p, i64, i64, i64, p, p, p, p, p, p]
        _LIB = L
    return _LIB


def polygonize(labels, n_regions):
    """Canonical rings of a label raster (the dm_polygonize contract) -> dict of ring_region int32, ring_offsets int64,
    ring_area int64, vertices int32 [n, 2], region_rings int64 [R + 1], counts int64 [4] (status counts[3] = 1 when a
    label >= n_regions; the arrays are then empty)."""
    import numpy as np
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    P = np.pad(L, 1, constant_values=-1)
    c = P[1:-1, 1:-1]
    sides = int(sum(((c >= 0) & (c != q)).sum() for q in (P[:-2, 1:-1], P[2:, 1:-1], P[1:-1, :-2], P[1:-1, 2:])))
    n = sides // 4 + 1
    rr, ro, ra = np.zeros(n, np.int32), np.zeros(n + 1, np.int64), np.zeros(n, np.int64)
    vt, reg, cnt = np.zeros((sides + 1, 2), np.int32), np.zeros(n_regions + 1, np.int64), np.zeros(4, np.int64)
    if lib().dmo_polygonize(L.ctypes.data, H, W, n_regions, rr.ctypes.data, ro.ctypes.data, ra.ctypes.data, vt.ctypes.data,
                            reg.ctypes.data, cnt.ctypes.data) != 0:
        raise MemoryError("dmo_polygonize")
    k, v = int(cnt[0]), int(cnt[1])
    return dict(ring_region=rr[:k].copy(), ring_offsets=ro[:k + 1].copy(), ring_area=ra[:k].copy(),
                vertices=vt[:v].copy(), region_rings=reg, counts=cnt)


def poly_successor(labels, x, y, side):
    """Successor of boundary side `side` of pixel (x, y) -> (x, y, side, corner), or None when it is not a boundary side."""
    import numpy as np
    L = np.ascontiguousarray(labels, np.int32)
    out = np.zeros(4, np.int64)
    if not lib().dmo_poly_successor(L.ctypes.data, L.shape[0], L.shape[1], x, y, side, out.ctypes.data):
        return None
    return tuple(int(v) for v in out)
