"""Loader of tests/lines_oracle.c, the sequential boundary-line tracer the tests and tools/time_lines.py compare dm_lines
against.  TEST INFRASTRUCTURE ONLY.  c_oracle.load builds it."""
from __future__ import annotations

import ctypes

from c_oracle import load


def lib():
    p, i64, i = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int
    return load("lines_oracle", {"dmo_line_segments": (i64, [p, i64, i64, p]),
                                 "dmo_lines": (i, [p, i64, i64, i64, p, p, p, p, p, p])})


def n_segments(L):
    import numpy as np
    v = np.pad(np.where(L >= 0, L, -1), 1, constant_values=-1)
    return int((v[1:, 1:-1] != v[:-1, 1:-1]).sum() + (v[1:-1, 1:] != v[1:-1, :-1]).sum())


def lines(labels, n_regions):
    """Canonical boundary lines of a label raster (the dm_lines contract) -> dict of line_left, line_right int32,
    line_length, line_offsets int64, vertices int32 [n, 2], counts int64 [4] (status counts[3] = 1 when a label
    >= n_regions; the arrays are then empty)."""
    import numpy as np
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    n = n_segments(L) + 1
    lf, rt, ln, off = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int64), np.zeros(n + 1, np.int64)
    vt, cnt = np.zeros((2 * n, 2), np.int32), np.zeros(4, np.int64)
    if lib().dmo_lines(L.ctypes.data, H, W, n_regions, lf.ctypes.data, rt.ctypes.data, ln.ctypes.data, off.ctypes.data,
                       vt.ctypes.data, cnt.ctypes.data) != 0:
        raise MemoryError("dmo_lines")
    k, v = int(cnt[0]), int(cnt[1])
    return dict(line_left=lf[:k].copy(), line_right=rt[:k].copy(), line_length=ln[:k].copy(),
                line_offsets=off[:k + 1].copy(), vertices=vt[:v].copy(), counts=cnt)


def segments(labels):
    """int64 [S, 9] per boundary segment: tail x, tail y, direction, head is a node, tail is a node, successor's tail
    x, y and direction (-1s at a node), head is a vertex of its line -- sorted by (tail y, tail x, direction)."""
    import numpy as np
    L = np.ascontiguousarray(labels, np.int32)
    H, W = L.shape
    out = np.zeros((n_segments(L) + 1, 9), np.int64)
    k = lib().dmo_line_segments(L.ctypes.data, H, W, out.ctypes.data)
    if k < 0:
        raise MemoryError("dmo_line_segments")
    out = out[:k]
    return out[np.lexsort((out[:, 2], out[:, 0], out[:, 1]))]
