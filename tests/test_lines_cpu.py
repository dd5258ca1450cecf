"""CPU: boundary lines of label rasters (dm_lines' contract, include/deepmerge_b200.h).

The sequential tracer of tests/lines_oracle.c (dmo_lines) is checked on the rasters of test_polygonize_cpu and on random
rasters with nodata against what shares no code with it: the boundary segments and vertex degrees counted by numpy, the
orientation rule, the canonical order, and the boundary lengths and perimeters of oracle_np.build_rag.  The shapefile
writer is checked by a round trip that pairs the line file with write_polygonized's polygon file.
deepmerge_b200/csrc/lines_core.cuh (the kernels' per-vertex rule) is compiled with g++ and checked against the oracle
on every 2 x 2 configuration.  The ABI rejects bad arguments without CUDA and before it enqueues anything (the checks
of tests/tracer_abi.py, which test_polygonize_cpu runs on dm_polygonize)."""
import ctypes
import itertools
import os
import subprocess

import numpy as np
import pytest

import lines_oracle as lo
import polygon_oracle as po
import tracer_abi
from oracle import oracle_np as o
from test_polygonize_cpu import CASES as POLY_CASES

HERE = os.path.dirname(os.path.abspath(__file__))
STEP = np.array([[1, 0], [0, 1], [-1, 0], [0, -1]], np.int64)       # directions 0 E, 1 S, 2 W, 3 N; y down


def _cases():
    c = dict(POLY_CASES)
    rng = np.random.default_rng(21)
    for i, (h, w, k) in enumerate([(1, 1, 2), (2, 2, 3), (7, 5, 4), (16, 23, 6), (40, 31, 3)]):
        L = rng.integers(-2, k, (h, w)).astype(np.int32)      # -2 is nodata too: its value is -1
        c["random_nodata_%d" % i] = (L, k)
    L, n = o.synth_labels(96, 80, 40, seed=3)
    L = L.copy()
    L[rng.random(L.shape) < 0.02] = -1
    L[30:50, 10:30] = -1
    c["voronoi_nodata"] = (L, n)
    c["island"] = (np.pad(np.full((3, 3), 1, np.int32), 2), 2)
    return c


CASES = _cases()


def values(L):
    """value of every pixel position, padded by one ring of -1 (index [y + 1, x + 1])"""
    return np.pad(np.where(L >= 0, L, -1), 1, constant_values=-1)


def segment_table(L):
    """(present bool [S_all], degree int [(H + 1), (W + 1)]) in the oracle's numbering of unit segments: horizontal
    ones y W + x for y in [0, H], then vertical ones (H + 1) W + y (W + 1) + x."""
    H, W = L.shape
    v = values(L)
    hor = v[:-1, 1:-1] != v[1:, 1:-1]            # [H + 1, W]: between (x, y - 1) and (x, y)
    ver = v[1:-1, :-1] != v[1:-1, 1:]            # [H, W + 1]: between (x - 1, y) and (x, y)
    deg = np.zeros((H + 1, W + 1), np.int64)
    deg[:, :-1] += hor
    deg[:, 1:] += hor
    deg[:-1, :] += ver
    deg[1:, :] += ver
    return np.concatenate([hor.ravel(), ver.ravel()]), deg


def expand(verts):
    """unit segments of a polyline: tail x, tail y, direction"""
    d = np.diff(verts.astype(np.int64), axis=0)
    n = np.abs(d).sum(1)
    assert ((d[:, 0] == 0) != (d[:, 1] == 0)).all(), "an edge is not axis-parallel or is empty"
    dirs = np.where(d[:, 0] > 0, 0, np.where(d[:, 1] > 0, 1, np.where(d[:, 0] < 0, 2, 3)))
    dd = np.repeat(dirs, n)
    first = np.repeat(np.cumsum(n) - n, n)
    k = np.arange(n.sum()) - first
    tails = np.repeat(verts[:-1].astype(np.int64), n, axis=0) + STEP[dd] * k[:, None]
    return tails[:, 0], tails[:, 1], dd


def check_invariants(L, R, P):
    """Every property of the contract that can be checked without another implementation."""
    H, W = L.shape
    lf, rt, ln, off, vt = P["line_left"], P["line_right"], P["line_length"], P["line_offsets"], P["vertices"]
    n = len(lf)
    assert P["counts"][3] == 0 and P["counts"][0] == n and P["counts"][1] == len(vt) == off[-1] and off[0] == 0
    present, deg = segment_table(L)
    assert P["counts"][2] == present.sum()
    if H == 0 or W == 0:
        assert n == 0
        return
    v = values(L)
    covered = np.zeros(present.shape, np.int64)
    keys = []
    pair_len, perim = {}, np.zeros(R, np.int64)
    for k in range(n):
        line = vt[off[k]:off[k + 1]].astype(np.int64)
        assert len(line) >= 2
        assert (line[:, 0] >= 0).all() and (line[:, 0] <= W).all() and (line[:, 1] >= 0).all() and (line[:, 1] <= H).all()
        tx, ty, d = expand(line)
        assert len(d) == ln[k]
        ids = np.where(d % 2 == 0, ty * W + np.where(d == 0, tx, tx - 1),
                       (H + 1) * W + np.where(d == 1, ty, ty - 1) * (W + 1) + tx)
        np.add.at(covered, ids, 1)
        # the values on the right / left of every unit segment (index into the padded raster: + 1)
        rx, ry = tx - ((d == 1) | (d == 2)), ty - ((d == 2) | (d == 3))
        lx, ly = tx - ((d == 2) | (d == 3)), ty - ((d == 0) | (d == 3))
        right, left = v[ry + 1, rx + 1], v[ly + 1, lx + 1]
        assert (right == rt[k]).all() and (left == lf[k]).all() and rt[k] > lf[k] >= -1
        # vertices: inner junctions of degree 2, corners only between the ends
        hx, hy = tx + STEP[d, 0], ty + STEP[d, 1]
        assert (deg[hy[:-1], hx[:-1]] == 2).all(), "a line runs through a node"
        turns = np.flatnonzero(d[1:] != d[:-1])
        assert np.array_equal(line[1:-1], np.stack([hx[turns], hy[turns]], 1)), "inner vertices are not the corners"
        start, end = tuple(line[0]), tuple(line[-1])
        if deg[start[1], start[0]] >= 3:
            assert deg[end[1], end[0]] >= 3, "an open line does not end at a node"
        else:
            assert start == end and d[0] != d[-1], "a closed line does not start at a corner"
            key = line[:, 1] * (W + 1) + line[:, 0]
            assert key[0] == key.min() and (key[:-1] == key[0]).sum() == 1, "closed line not at its smallest vertex"
        keys.append((int(line[0, 1]), int(line[0, 0]), int(d[0])))
        if lf[k] >= 0:
            pk = (int(lf[k]), int(rt[k]))
            pair_len[pk] = pair_len.get(pk, 0) + int(ln[k])
            perim[lf[k]] += ln[k]
        perim[rt[k]] += ln[k]
    assert np.array_equal(covered, present.astype(np.int64)), "boundary segments not covered exactly once"
    assert keys == sorted(keys) and len(set(keys)) == n, "lines out of canonical order"
    ekeys, blen, _, per = o.build_rag(L, R)
    got = sorted(((a << 32) | b, m) for (a, b), m in pair_len.items())
    assert [k for k, _ in got] == ekeys.tolist() and [m for _, m in got] == blen.tolist()
    assert np.array_equal(perim, per)


@pytest.mark.parametrize("name", sorted(CASES))
def test_oracle_invariants(name):
    L, R = CASES[name]
    check_invariants(L, R, lo.lines(L, R))


def test_known_lines():
    # two regions side by side: the nodes (1, 0) and (1, 2) split the boundary into one line between them (region 1 on
    # the right: north) and one along the border of each region
    P = lo.lines(np.array([[0, 1], [0, 1]], np.int32), 2)
    assert P["line_left"].tolist() == [-1, -1, 0] and P["line_right"].tolist() == [1, 0, 1]
    assert P["vertices"].tolist() == [[1, 0], [2, 0], [2, 2], [1, 2], [1, 2], [0, 2], [0, 0], [1, 0], [1, 2], [1, 0]]
    assert P["line_length"].tolist() == [4, 4, 2]
    # an island: one closed line each, starting at the smallest vertex and closed by repeating it
    L, R = CASES["island"]
    P = lo.lines(L, R)
    assert P["line_left"].tolist() == [-1, 0] and P["line_right"].tolist() == [0, 1]
    island = P["vertices"][P["line_offsets"][1]:P["line_offsets"][2]].tolist()
    assert island == [[2, 2], [5, 2], [5, 5], [2, 5], [2, 2]]      # region 1 (larger) on the right: east first
    # a saddle is a node: four single-segment lines meet there
    P = lo.lines(np.array([[0, 1], [1, 0]], np.int32), 2)
    assert P["counts"][0] == 8 and sorted(P["line_length"].tolist()) == [1, 1, 1, 1, 2, 2, 2, 2]


def test_label_out_of_range_is_reported():
    assert lo.lines(np.array([[0, 5]], np.int32), 2)["counts"][3] == 1


# ---- the write path -------------------------------------------------------------------------------------------------

def as_lines(P):
    import torch
    from deepmerge_b200 import Lines
    t = torch.from_numpy
    return Lines(t(P["line_left"]), t(P["line_right"]), t(P["line_length"]), t(P["line_offsets"]), t(P["vertices"]),
                 int(P["counts"][2]))


def check_write_path(L, R, P, tmp_path):
    """write_boundary_lines -> read_polylines + DbfTable: geometry, LENGTH, and LEFT_FID / RIGHT_FID equal to the record
    indices of write_polygonized on the same raster, with the right-hand region on the right in map coordinates."""
    from test_polygonize_cpu import as_polygons
    from deepmerge_b200 import shapefile as shp
    polys = as_polygons(po.polygonize(L, R))
    lines = as_lines(P)
    for i, gt in enumerate([(500.0, 2.0, 0.0, 9000.0, 0.0, -2.0), (-30.0, 0.5, 0.0, 10.0, 0.0, 0.25)]):
        lpath, ppath = str(tmp_path / ("lines%d.shp" % i)), str(tmp_path / ("poly%d.shp" % i))
        shp.write_boundary_lines(lpath, lines, gt)
        shp.write_polygonized(ppath, polys, gt)
        assert shp.shape_type(lpath) == 3
        region = shp.DbfTable(ppath[:-4] + ".dbf").column_int("REGION")
        t = shp.DbfTable(lpath[:-4] + ".dbf")
        lfid, rfid = t.column_int("LEFT_FID"), t.column_int("RIGHT_FID")
        assert np.array_equal(t.column_int("LENGTH"), P["line_length"])
        assert np.array_equal(np.where(lfid >= 0, region[lfid], -1), P["line_left"])
        assert np.array_equal(region[rfid], P["line_right"])
        geoms = shp.read_polylines(lpath)
        assert len(geoms) == len(P["line_left"])
        off = P["line_offsets"]
        for k, parts in enumerate(geoms):
            assert len(parts) == 1
            xy = parts[0]
            pix = np.stack([(xy[:, 0] - gt[0]) / gt[1], (xy[:, 1] - gt[3]) / gt[5]], 1)
            want = P["vertices"][off[k]:off[k + 1]]
            assert np.array_equal(pix, want if gt[1] * gt[5] < 0 else want[::-1])
            # just after the start, a quarter pixel to the right / left of travel in map coordinates (X east, Y north:
            # the right of (ex, ey) is (ey, -ex)) lies the pixel of RIGHT_FID / LEFT_FID
            e = (xy[1] - xy[0]) / np.linalg.norm(xy[1] - xy[0])
            eps = 0.25 * min(abs(gt[1]), abs(gt[5]))
            for sign, fids in ((1, rfid), (-1, lfid)):
                q = xy[0] + eps * e + sign * eps * np.array([e[1], -e[0]])
                px, py = int(np.floor((q[0] - gt[0]) / gt[1])), int(np.floor((q[1] - gt[3]) / gt[5]))
                inside = 0 <= px < L.shape[1] and 0 <= py < L.shape[0]
                got = L[py, px] if inside and L[py, px] >= 0 else -1
                assert got == (region[fids[k]] if fids[k] >= 0 else -1), (k, sign)


@pytest.mark.parametrize("name", ["two_pieces", "hole_with_island", "speckle_nodata", "voronoi_nodata", "saddle_self"])
def test_write_path_round_trip(name, tmp_path):
    L, R = CASES[name]
    check_write_path(L, R, lo.lines(L, R), tmp_path)


def test_shapes_rejects_rotated_geotransform():
    lines = as_lines(lo.lines(np.zeros((2, 2), np.int32), 1))
    with pytest.raises(ValueError):
        lines.shapes((0.0, 1.0, 0.5, 0.0, 0.0, -1.0))


# ---- lines_core.cuh against the oracle's rule -----------------------------------------------------------------------

@pytest.fixture(scope="module")
def core(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("lines_core") / "liblines_core_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", so,
                        os.path.join(HERE, "lines_core_host.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(so)
    lib.line_core_segments.restype = ctypes.c_long
    lib.line_core_segments.argtypes = [ctypes.c_void_p, ctypes.c_long, ctypes.c_long, ctypes.c_long, ctypes.c_void_p]

    def run(L):
        L = np.ascontiguousarray(L, np.int32)
        H, W = L.shape
        out = np.full((H * W * 4, 9), -2, np.int64)
        n = lib.line_core_segments(L.ctypes.data, H, W, W, out.ctypes.data)
        assert n >= 0, "a successor is not owned where owner_of says"
        out = out[out[:, 0] != -2]
        assert len(out) == n
        return out[np.lexsort((out[:, 2], out[:, 0], out[:, 1]))]
    return run


def test_core_rule_on_every_2x2_block(core):
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
            got, want = core(r), lo.segments(r)
            assert np.array_equal(got, want), (blk, r)
            n_checked += len(got)
    assert n_checked > 10000


# ---- ABI without CUDA -----------------------------------------------------------------------------------------------

def test_abi_rejects_bad_arguments_without_cuda():
    tracer_abi.check_rejects_bad_arguments("dm_lines")


def test_no_work_is_enqueued_before_an_argument_error():
    tracer_abi.check_no_work_before_an_argument_error("dm_lines")


def test_boundary_lines_refuses_cpu_tensors():
    import torch
    from deepmerge_b200 import boundary_lines
    with pytest.raises(ValueError):
        boundary_lines(torch.zeros((4, 4), dtype=torch.int32), 2)
