"""CPU: simplified rings and lines (dm_polygonize_simplified / dm_lines_simplified, include/deepmerge_b200.h).

deepmerge_b200/csrc/simplify_core.cuh (the kernels' distance comparison, top-vertex order and tolerance rounding) is
compiled with g++ and checked against the independent arithmetic of the sequential simplifier tests/simplify_oracle.c.
The oracle is checked against the contract's consequences on the rasters of test_lines_cpu / test_polygonize_cpu and on
Voronoi maps: kept vertices are an ordered subset holding every anchor, every dropped vertex lies within t of its output
segment, reversal commutes with simplification, kept sets shrink as t grows, every ring is the concatenation of the
simplified lines around it, no ring falls below 3 distinct vertices, and the ring areas add up to the raster.  The ABI
rejects bad tolerances and extents without CUDA and before it enqueues anything."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import simplify_oracle as so
from oracle import oracle_np as o
from test_lines_cpu import CASES as LINE_CASES

HERE = os.path.dirname(os.path.abspath(__file__))
TOLERANCES = (0.0, 0.5, 1.0, 1.5, 4.0, 1e9)


def _cases():
    c = dict(LINE_CASES)
    for i, (h, w, k) in enumerate([(64, 64, 30), (37, 91, 12), (120, 80, 200)]):
        c["voronoi_%d" % i] = o.synth_labels(h, w, k, seed=40 + i)
    return c


CASES = _cases()


@pytest.fixture(scope="module")
def core(tmp_path_factory):
    so_path = str(tmp_path_factory.mktemp("simplify_core") / "libsimplify_core_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so_path,
                        os.path.join(HERE, "simplify_core_host.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    L = ctypes.CDLL(so_path)
    L.core_top.restype = ctypes.c_long
    L.core_top.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_uint64, ctypes.c_void_p]
    L.core_quantize.restype = ctypes.c_uint64
    L.core_quantize.argtypes = [ctypes.c_double, ctypes.c_long, ctypes.c_long]
    return L


def _oracle_top():
    L = so.lib()
    L.dmo_top.restype = ctypes.c_int64
    L.dmo_top.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_uint64, ctypes.c_void_p]
    L.dmo_quantize.restype = ctypes.c_uint64
    L.dmo_quantize.argtypes = [ctypes.c_double, ctypes.c_int64, ctypes.c_int64]
    return L


def _tops(lib, fn, v, W, T):
    v = np.ascontiguousarray(v, np.int32)
    ex = ctypes.c_int(0)
    k = getattr(lib, fn)(v.ctypes.data, len(v) - 1, W, T, ctypes.byref(ex))
    return int(k), int(ex.value)


@pytest.mark.parametrize("kind", ["random", "ties", "closed", "largest_extent"])
def test_core_matches_oracle(core, kind):
    rng = np.random.default_rng(hash(kind) % 2**32)
    ol = _oracle_top()
    top = (1 << 26) - 1
    for _ in range(3000):
        n = int(rng.integers(2, 40))
        if kind == "largest_extent":
            W = top
            v = rng.choice([0, 1, 2, top - 2, top - 1, top], size=(n + 1, 2)).astype(np.int64)
            v[rng.random(n + 1) < 0.5] = rng.integers(0, top + 1, (2,))
        else:
            span = 4 if kind == "ties" else 200
            W = span
            v = rng.integers(0, span + 1, (n + 1, 2))
        if kind == "closed":
            v[-1] = v[0]
        T = int(rng.choice([0, 1, 512, 1024, 1536, 4096, int(rng.integers(0, 1 << 20)), (2 * W) << 10]))
        assert _tops(core, "core_top", v, W, T) == _tops(ol, "dmo_top", v, W, T), (v.tolist(), T)


def test_tolerance_rounding(core):
    ol = _oracle_top()
    for t in [0.0, 1e-4, 0.4999 / 1024, 0.5 / 1024, 1.5 / 1024, 0.5, 1.0, 1.5, 3.7, 99.99, 1e9, 2.0 ** 40]:
        for H, W in [(10, 20), (1, 1), ((1 << 26) - 1, (1 << 26) - 1)]:
            assert core.core_quantize(t, H, W) == ol.dmo_quantize(t, H, W) == int(np.floor(min(t, H + W) * 1024 + 0.5))


# --- the oracle against the contract ---------------------------------------------------------------------------

def _seg_dist(p, a, b):
    p, a, b = (np.asarray(z, np.float64) for z in (p, a, b))
    v, w = b - a, p - a
    vv = v @ v
    if vv == 0:
        return float(np.hypot(*w))
    s = min(max((w @ v) / vv, 0.0), 1.0)
    return float(np.hypot(*(w - s * v)))


def _chains(off):
    return [(int(off[k]), int(off[k + 1])) for k in range(len(off) - 1)]


def _anchors(v, lo, hi, H, W, cyclic, node):
    x, y = v[lo:hi, 0], v[lo:hi, 1]
    a = (x == 0) | (y == 0) | (x == W) | (y == H)
    if cyclic:
        nd = node[lo:hi].astype(bool)
        a |= nd
        if not nd.any():
            a[0] = True
    else:
        a[0] = a[-1] = True
    return a


def _check_chains(v, off, keep, H, W, t, cyclic, node=None):
    tq = min(np.floor(min(t, H + W) * 1024 + 0.5) / 1024, H + W)
    for lo, hi in _chains(off):
        k = keep[lo:hi]
        assert k[_anchors(v, lo, hi, H, W, cyclic, node)].all(), "an anchor was dropped"
        idx = np.flatnonzero(k)
        # every dropped vertex within t of the output segment that replaced it
        n = hi - lo
        ends = list(zip(idx, np.r_[idx[1:], idx[0] + n])) if cyclic else list(zip(idx[:-1], idx[1:]))
        for a, b in ends:
            A, B = v[lo + a % n], v[lo + b % n]
            for j in range(a + 1, b):
                assert _seg_dist(v[lo + j % n], A, B) <= tq + 1e-9, "a dropped vertex is farther than t"
        if cyclic:
            kept = {tuple(p) for p in v[lo:hi][k]}
            assert len(kept) >= 3, "a ring has fewer than 3 distinct vertices"


def _line_table(lv, loff, lkeep):
    """full vertex tuple -> kept vertex tuple, for every line forward and reversed"""
    table = {}
    for lo, hi in _chains(loff):
        full, kept = lv[lo:hi], lv[lo:hi][lkeep[lo:hi]]
        table[tuple(map(tuple, full))] = tuple(map(tuple, kept))
        table[tuple(map(tuple, full[::-1]))] = tuple(map(tuple, kept[::-1]))
    return table


def _check_rings_are_lines(rv, roff, rnode, rkeep, table):
    for lo, hi in _chains(roff):
        n = hi - lo
        nodes = np.flatnonzero(rnode[lo:hi])
        cuts = [(0, n)] if len(nodes) == 0 else [(a, b) for a, b in zip(nodes, np.r_[nodes[1:], nodes[0] + n])]
        for a, b in cuts:
            pos = [lo + j % n for j in range(a, b + 1)]
            full = tuple(map(tuple, rv[pos]))
            assert full in table, "a ring piece is no line"
            kept = tuple(map(tuple, rv[[p for p in pos if rkeep[p]]]))
            assert kept == table[full], "a ring piece is not simplified as its line"


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_contract(name):
    L, R = CASES[name]
    H, W = L.shape
    if H == 0 or W == 0:
        return
    prev = None
    for t in TOLERANCES:
        P = so.polygons(L, R, t)
        Q = so.lines(L, R, t)
        rv, roff, rnode = P["full"]
        lv, loff = Q["full"]
        rkeep = so.keep(rv, roff, H, W, t, rnode)
        lkeep = so.keep(lv, loff, H, W, t)
        _check_chains(rv, roff, rkeep, H, W, t, True, rnode)
        _check_chains(lv, loff, lkeep, H, W, t, False)
        # reversal: every line reversed, simplified, gives the reversed result
        rev = np.concatenate([lv[lo:hi][::-1] for lo, hi in _chains(loff)]) if len(loff) > 1 else lv
        rk = so.keep(rev, loff, H, W, t)
        assert np.array_equal(np.concatenate([rk[lo:hi][::-1] for lo, hi in _chains(loff)]) if len(loff) > 1 else rk,
                              lkeep)
        # kept sets shrink as t grows
        if prev is not None:
            assert not (rkeep & ~prev[0]).any() and not (lkeep & ~prev[1]).any()
        prev = (rkeep, lkeep)
        _check_rings_are_lines(rv, roff, rnode, rkeep, _line_table(lv, loff, lkeep))
        # the outputs: ordered subsets with their offsets
        assert np.array_equal(P["vertices"], rv[rkeep]) and P["ring_offsets"][-1] == rkeep.sum()
        assert np.array_equal(Q["vertices"], lv[lkeep]) and Q["line_offsets"][-1] == lkeep.sum()
        if (L >= 0).all() and R > int(L.max()):
            assert ring_area_sum(P["vertices"], P["ring_offsets"]) == 2 * H * W


def ring_area_sum(v, off):
    """sum over rings of the doubled signed shoelace area"""
    v = v.astype(np.int64)
    total = 0
    for lo, hi in _chains(off):
        x, y = v[lo:hi, 0], v[lo:hi, 1]
        total += int((x * np.roll(y, -1) - np.roll(x, -1) * y).sum())
    return total


def test_nodes_are_added_where_a_ring_goes_straight():
    # region 0 above a boundary that regions 1 and 2 meet below: (2, 2) is a node on a straight side of region 0
    L = np.array([[0, 0, 0, 0], [0, 0, 0, 0], [1, 1, 2, 2], [1, 1, 2, 2]], np.int32)
    P = so.polygons(L, 3, 1e9)
    v, off, node = P["full"]
    assert (2, 2) in {tuple(p) for p, f in zip(v, node) if f}
    ring0 = P["vertices"][P["ring_offsets"][0]:P["ring_offsets"][1]]
    assert (2, 2) in {tuple(p) for p in ring0}


# --- ABI -----------------------------------------------------------------------------------------------------------

ENTRIES = {
    "dm_polygonize_simplified": (lambda L, H, W, R, cap: L.dm_polygonize_simplified_workspace_bytes(H, W, R, cap), 5),
    "dm_lines_simplified": (lambda L, H, W, R, cap: L.dm_lines_simplified_workspace_bytes(H, W, cap), 5),
}


@pytest.mark.parametrize("entry", sorted(ENTRIES))
def test_abi_rejects_bad_tolerance_and_extent(entry):
    from deepmerge_b200 import _lib
    L = _lib.lib()
    bad, short = _lib.DM_ERR_BAD_ARG, _lib.DM_ERR_WORKSPACE
    f = getattr(L, entry)
    wsq, n_out = ENTRIES[entry]
    nul = [None] * n_out
    ws = wsq(L, 4, 4, 3, 64)
    assert ws > 0
    fake = 16      # an address nothing may dereference: every CUDA call would fail there first
    for t in (float("nan"), float("inf"), float("-inf"), -1e-9, -1.0):
        n0 = L.dm_launch_count()
        assert f(fake, 4, 4, 4, 3, 64, t, *[fake] * n_out, fake, fake, ws, None) == bad, t
        assert f(None, 0, 4, 4, 3, 64, t, *nul, None, None, 0, None) == bad, t        # also for the empty raster
        assert L.dm_launch_count() == n0
    n0 = L.dm_launch_count()
    assert f(fake, 4, 4, 4, 3, 64, 1.0, *[fake] * n_out, fake, fake, ws - 1, None) == short
    assert f(fake, 4, 4, 3, 3, 64, 1.0, *[fake] * n_out, fake, fake, ws, None) == bad                  # ld < W
    assert f(fake, 1, 1 << 26, 1 << 26, 3, 64, 1.0, *[fake] * n_out, fake, fake, ws, None) == bad      # W >= 2^26
    assert f(fake, 1 << 26, 1, 1, 3, 64, 1.0, *[fake] * n_out, fake, fake, ws, None) == bad            # H >= 2^26
    assert f(None, 4, 4, 4, 3, 64, 1.0, *nul, None, None, 0, None) == bad                              # null pointers
    assert L.dm_launch_count() == n0
    assert f(None, 0, 4, 4, 3, 64, 1.0, *nul, None, None, 0, None) == 0                                # empty raster
    assert f(None, 4, 0, 0, 3, 64, 0.0, *nul, None, None, 0, None) == 0
    assert wsq(L, 1, 1 << 26, 3, 64) == 0 and wsq(L, 64, 64, 3, -1) == 0
    assert 0 < wsq(L, 64, 64, 3, 1000) < wsq(L, 64, 64, 3, 100000)


def test_python_rejects_bad_tolerance():
    from deepmerge_b200.polygons import _tolerance
    for t in (float("nan"), float("inf"), -1.0):
        with pytest.raises(ValueError):
            _tolerance(t)
    assert _tolerance(None) == () and _tolerance(2) == (2.0,)
