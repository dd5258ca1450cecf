"""CPU: polygonizing label rasters (dm_polygonize's contract, include/deepmerge_b200.h).

The sequential tracer of tests/polygon_oracle.c (dmo_polygonize) is checked on hand-made and random rasters against
what shares no code with it: the round trip through the shapefile writer / reader and rasterize_polygons, the pixel counts and the
perimeters of oracle_np.build_rag.  deepmerge_b200/csrc/polygon_core.cuh (the kernels' per-side rule) is compiled with
g++ and checked against the oracle's successor rule on every 2 x 2 configuration.  The ABI rejects bad arguments without
CUDA and before it enqueues anything (the checks of tests/tracer_abi.py, which test_lines_cpu runs on dm_lines)."""
import ctypes
import itertools
import os
import subprocess

import numpy as np
import pytest

import polygon_oracle as po
import tracer_abi
from oracle import oracle_np as o

HERE = os.path.dirname(os.path.abspath(__file__))


def _hole_with_island():
    L = np.full((9, 9), 1, np.int32)
    L[2:7, 2:7] = 0          # region 0 ...
    L[3:6, 3:6] = 2          # ... with a hole of region 2 ...
    L[4, 4] = 0              # ... that holds an island of region 0
    return L, 3


def _saddle_self():
    # region 0 reaches around and touches itself diagonally at the vertex (2, 2) (pixels (1, 1) and (2, 2))
    L = np.array([[0, 0, 0, 0],
                  [0, 0, 1, 0],
                  [0, 1, 0, 0],
                  [0, 0, 0, 0]], np.int32)
    return L, 2


def _cases():
    rng = np.random.default_rng(7)
    c = {
        "single_pixel": (np.zeros((1, 1), np.int32), 1),
        "row_strip": (np.array([[0, 0, 1, 1, 0, 2, -1, 2]], np.int32), 3),
        "column_strip": (np.array([[0], [0], [1], [-1], [1], [1]], np.int32), 2),
        "filled": (np.full((5, 7), 3, np.int32), 4),
        "all_nodata": (np.full((4, 5), -1, np.int32), 2),
        "empty_rows": (np.zeros((0, 5), np.int32), 1),
        "empty_cols": (np.zeros((5, 0), np.int32), 1),
        "checkerboard": ((np.add.outer(np.arange(8), np.arange(9)) % 2).astype(np.int32), 2),
        "speckle": (rng.integers(0, 3, (23, 29)).astype(np.int32), 3),
        "speckle_nodata": (rng.integers(-1, 3, (31, 17)).astype(np.int32), 3),
        "hole_with_island": _hole_with_island(),
        "two_pieces": (np.array([[0, 0, 1, 1, 0], [0, 1, 1, 1, 0], [1, 1, 2, 1, 0]], np.int32), 3),
        "saddle_self": _saddle_self(),
    }
    L = np.zeros((6, 6), np.int32)
    L[2:4, 2:4] = -1
    c["nodata_hole"] = (L, 1)
    sl, n = o.synth_labels(256, 256, 300, seed=11)
    c["voronoi"] = (sl, n)
    return c


CASES = _cases()


def shoelace2(v):
    x, y = v[:, 0].astype(np.int64), v[:, 1].astype(np.int64)
    return int((x * np.roll(y, -1) - np.roll(x, -1) * y).sum())


def check_invariants(L, R, P):
    """Every property of the contract that can be checked without another implementation."""
    H, W = L.shape
    rr, ro, ra, v, reg = P["ring_region"], P["ring_offsets"], P["ring_area"], P["vertices"], P["region_rings"]
    n = len(rr)
    assert P["counts"][3] == 0 and P["counts"][0] == n and P["counts"][1] == len(v) == ro[-1] and ro[0] == 0
    valid = L[L >= 0]
    assert np.array_equal(reg, np.concatenate([[0], np.cumsum(np.bincount(rr, minlength=R))]))
    area = np.zeros(R, np.int64)
    np.add.at(area, rr, ra)
    assert np.array_equal(area, np.bincount(valid, minlength=R)), "sum of ring areas != pixel count"
    per = np.zeros(R, np.int64)
    starts = []
    for k in range(n):
        ring = v[ro[k]:ro[k + 1]].astype(np.int64)
        m = len(ring)
        assert m >= 4 and m % 2 == 0
        assert (ring[:, 0] >= 0).all() and (ring[:, 0] <= W).all() and (ring[:, 1] >= 0).all() and (ring[:, 1] <= H).all()
        d = np.roll(ring, -1, axis=0) - ring
        horiz = d[:, 1] == 0
        assert ((d[:, 0] == 0) != horiz).all(), "an edge is not axis-parallel or is empty"
        assert (horiz != np.roll(horiz, -1)).all(), "edges do not alternate (a vertex is not a corner)"
        per[rr[k]] += int(np.abs(d).sum())
        assert shoelace2(ring) == 2 * ra[k]
        key = ring[:, 1] * (W + 1) + ring[:, 0]
        assert key[0] == key.min() and (key == key[0]).sum() == 1, "ring does not start at its unique smallest vertex"
        starts.append((int(rr[k]), int(ring[0, 1]), int(ring[0, 0])))
    assert starts == sorted(starts) and len(set(starts)) == len(starts), "rings out of canonical order"
    if H and W:
        _, _, _, perim = o.build_rag(L, R)
        assert np.array_equal(per, perim), "ring lengths != perimeter"
    else:
        assert n == 0


def as_polygons(P):
    import torch
    from deepmerge_b200 import Polygons
    t = torch.from_numpy
    return Polygons(t(P["ring_region"]), t(P["ring_offsets"]), t(P["ring_area"]), t(P["vertices"]), t(P["region_rings"]),
                    int(P["counts"][2]))


def check_round_trip(L, P, tmp_path, columns=None):
    """Polygons.shapes -> write_polygonized -> read_polygons -> rasterize_polygons(ids = REGION) == labels, for a
    north-up and a south-up geotransform; outer rings clockwise and holes counter-clockwise in the file."""
    from deepmerge_b200 import shapefile as shp
    H, W = L.shape
    polys = as_polygons(P)
    for i, gt in enumerate([(500.0, 2.0, 0.0, 9000.0, 0.0, -2.0), (-30.0, 0.5, 0.0, 10.0, 0.0, 0.25)]):
        path = str(tmp_path / ("poly%d.shp" % i))
        shp.write_polygonized(path, polys, gt, columns)
        rings = shp.read_polygons(path)
        table = shp.DbfTable(path[:-4] + ".dbf")
        ids = table.column_int("REGION")
        assert list(ids) == sorted(set(ids.tolist())) == sorted(set(P["ring_region"].tolist()))
        area = table.column_int("AREA")
        assert np.array_equal(area, np.bincount(L[L >= 0], minlength=int(ids.max(initial=-1)) + 1)[ids])
        back = shp.rasterize_polygons(rings, gt, H, W, nodata=-1, ids=ids)
        assert np.array_equal(back, np.where(L >= 0, L, -1))
        # orientation in map coordinates: clockwise (negative shoelace with Y up) for outer rings, holes the other way
        rr, ra, reg = P["ring_region"], P["ring_area"], P["region_rings"]
        for rec, rid in enumerate(ids):
            for j, ring in enumerate(rings[rec]):
                assert np.array_equal(ring[0], ring[-1])
                xy = ring[:-1]
                a = 0.5 * float((xy[:, 0] * np.roll(xy[:, 1], -1) - np.roll(xy[:, 0], -1) * xy[:, 1]).sum())
                k = reg[rid] + j
                assert rr[k] == rid and np.sign(a) == -np.sign(ra[k])
        if columns:
            for name, col in columns.items():
                assert np.allclose(table.column_float(name), np.asarray(col)[ids])


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_invariants_and_round_trip(name, tmp_path):
    L, R = CASES[name]
    P = po.polygonize(L, R)
    check_invariants(L, R, P)
    if L.size:
        check_round_trip(L, P, tmp_path)


def test_known_rings():
    P = po.polygonize(np.array([[0, 0], [0, 1]], np.int32), 2)
    assert P["ring_region"].tolist() == [0, 1]
    assert P["vertices"].tolist() == [[0, 0], [2, 0], [2, 1], [1, 1], [1, 2], [0, 2], [1, 1], [2, 1], [2, 2], [1, 2]]
    assert P["ring_area"].tolist() == [3, 1]
    # a hole: the outer ring runs east first, the hole ring (region on its right) south first, with negative area
    L, R = _hole_with_island()
    P = po.polygonize(L, R)
    r0 = slice(P["region_rings"][0], P["region_rings"][1])
    assert P["ring_area"][r0].tolist() == [25, -9, 1]
    hole = P["vertices"][P["ring_offsets"][1]:P["ring_offsets"][2]]
    assert hole[:2].tolist() == [[3, 3], [3, 6]]
    # the saddle: region 0 is one outer ring that passes the vertex (2, 2) twice, region 1 is two pieces
    L, R = _saddle_self()
    P = po.polygonize(L, R)
    assert P["ring_region"].tolist() == [0, 0, 1, 1] and P["ring_area"].tolist() == [16, -2, 1, 1]
    inner = P["vertices"][P["ring_offsets"][1]:P["ring_offsets"][2]].tolist()
    assert inner.count([2, 2]) == 2


def test_label_out_of_range_is_reported():
    P = po.polygonize(np.array([[0, 5]], np.int32), 2)
    assert P["counts"][3] == 1


def test_columns_are_written(tmp_path):
    L, R = CASES["two_pieces"]
    P = po.polygonize(L, R)
    check_round_trip(L, P, tmp_path, columns={"PERI": o.build_rag(L, R)[3], "SCORE": np.array([0.5, 1.25, -2.0])})


def test_shapes_rejects_rotated_geotransform():
    polys = as_polygons(po.polygonize(np.zeros((2, 2), np.int32), 1))
    with pytest.raises(ValueError):
        polys.shapes((0.0, 1.0, 0.5, 0.0, 0.0, -1.0))


# ---- polygon_core.cuh against the oracle's successor rule ---------------------------------------------------------

@pytest.fixture(scope="module")
def core(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("polygon_core") / "libpolygon_core_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                        os.path.join(HERE, "polygon_core_host.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(so)
    lib.poly_core_successors.restype = ctypes.c_long
    lib.poly_core_successors.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_long, ctypes.c_void_p]

    def run(L):
        L = np.ascontiguousarray(L, np.int32)
        H, W = L.shape
        out = np.zeros((H, W, 4, 4), np.int64)
        n = lib.poly_core_successors(L.ctypes.data, H, W, W, out.ctypes.data)
        return n, out
    return run


def oracle_successors(L):
    H, W = L.shape
    out = np.full((H, W, 4, 4), -1, np.int64)
    for y in range(H):
        for x in range(W):
            for s in range(4):
                q = po.poly_successor(L, x, y, s)
                if q is not None:
                    out[y, x, s] = q
    return out


def test_core_successor_rule_on_every_2x2_block(core):
    """All 5^4 blocks over {nodata, a, b, c, d}: alone (the image border on every side), and placed in each corner and
    the middle of a 4 x 4 raster (border on two sides / none), whose other pixels are a fixed label pattern."""
    vals = [-1, 0, 1, 2, 3]
    rng = np.random.default_rng(3)
    fill = rng.integers(-1, 4, (4, 4)).astype(np.int32)
    n_checked = 0
    for blk in itertools.product(vals, repeat=4):
        b = np.array(blk, np.int32).reshape(2, 2)
        rasters = [b]
        for y0, x0 in ((0, 0), (0, 2), (2, 0), (2, 2), (1, 1)):
            r = fill.copy()
            r[y0:y0 + 2, x0:x0 + 2] = b
            rasters.append(r)
        for r in rasters:
            n, got = core(r)
            want = oracle_successors(r)
            assert np.array_equal(got, want), (blk, r)
            n_checked += n
    assert n_checked > 10000


# ---- ABI without CUDA -----------------------------------------------------------------------------------------------

def test_abi_rejects_bad_arguments_without_cuda():
    tracer_abi.check_rejects_bad_arguments("dm_polygonize")


def test_no_work_is_enqueued_before_an_argument_error():
    tracer_abi.check_no_work_before_an_argument_error("dm_polygonize")


def test_polygonize_refuses_cpu_tensors():
    import torch
    from deepmerge_b200 import polygonize
    with pytest.raises(ValueError):
        polygonize(torch.zeros((4, 4), dtype=torch.int32), 2)
