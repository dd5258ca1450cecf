"""CPU: the polygon rasterizer (dm_rasterize).

deepmerge_b200/csrc/rasterize_core.cuh holds the per-segment arithmetic the kernels call; the same header is compiled
here with g++ -ffp-contract=off (tests/rasterize_core_host.cpp) and checked bit for bit against numpy's own expressions
from shapefile.rasterize_polygons: the pixel transform, the crossing predicate, the exact set of rows a segment crosses,
the crossing x and its column.  The flat reader shapefile.read_polygon_rings is checked against read_polygons and a
record-by-record restatement of the .shp layout, and the C ABI's argument checks run without CUDA."""
import ctypes
import os
import struct
import subprocess

import numpy as np
import pytest

from deepmerge_b200 import shapefile

HERE = os.path.dirname(os.path.abspath(__file__))
D = ctypes.c_void_p


@pytest.fixture(scope="module")
def core(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("rasterize_core") / "librasterize_core_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                        os.path.join(HERE, "rasterize_core_host.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(so)


def _f(a):
    a = np.ascontiguousarray(a, np.float64)
    return a, a.ctypes.data


def pixel(core, v, origin, size):
    v, p = _f(v)
    out = np.empty_like(v)
    core.pixel_host(D(p), ctypes.c_long(len(v)), ctypes.c_double(origin), ctypes.c_double(size), D(out.ctypes.data))
    return out


def rows(core, y0, y1, H):
    (y0, p0), (y1, p1) = _f(y0), _f(y1)
    first, count = np.empty(len(y0), np.int64), np.empty(len(y0), np.int64)
    core.rows_host(D(p0), D(p1), ctypes.c_long(len(y0)), ctypes.c_long(H), D(first.ctypes.data), D(count.ctypes.data))
    return first, count


def xi(core, x0, y0, x1, y1, yc):
    arrs = [_f(a) for a in (x0, y0, x1, y1, yc)]
    out = np.empty(len(arrs[0][0]))
    core.xi_host(*[D(p) for _, p in arrs], ctypes.c_long(len(out)), D(out.ctypes.data))
    return out


def col(core, x, W):
    x, p = _f(x)
    out = np.empty(len(x), np.int64)
    core.col_host(D(p), ctypes.c_long(len(x)), ctypes.c_long(W), D(out.ctypes.data))
    return out


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def segments(rng, n, H, W):
    """Segments in pixel coordinates around a raster of H x W: random, on row centres (yc == y0 or y1), vertical on
    column centres and at pixel corners (xi - 0.5 an integer), horizontal, and huge and tiny coordinates."""
    k = n // 8
    y0 = rng.uniform(-8, H + 8, n)
    y1 = y0 + rng.normal(0, rng.choice([0.3, 3, 30], n))
    x0 = rng.uniform(-8, W + 8, n)
    x1 = x0 + rng.normal(0, rng.choice([0.3, 3, 30], n))
    y0[:k] = rng.integers(-2, H + 2, k) + 0.5                   # starts on a row centre
    y1[k:2 * k] = rng.integers(-2, H + 2, k) + 0.5              # ends on one
    x0[2 * k:3 * k] = rng.integers(-2, W + 2, k) + 0.5          # vertical, on a column centre: xi - 0.5 an integer
    x1[2 * k:3 * k] = x0[2 * k:3 * k]
    x0[3 * k:4 * k] = rng.integers(-2, W + 2, k).astype(float)  # vertical on a pixel corner
    x1[3 * k:4 * k] = x0[3 * k:4 * k]
    y1[4 * k:5 * k] = y0[4 * k:5 * k]                           # horizontal
    y0[4 * k:4 * k + k // 2] = np.round(y0[4 * k:4 * k + k // 2]) + 0.5
    y1[4 * k:4 * k + k // 2] = y0[4 * k:4 * k + k // 2]
    huge = rng.choice([1e15, 1e100, 1e300, 2.0 ** 52, 2.0 ** 53 + 1], k) * rng.choice([-1, 1], k)
    y0[5 * k:6 * k] = huge                                       # one end far away
    x1[5 * k:6 * k] = huge[::-1]
    tiny = rng.choice([1e-300, 5e-324, 1e-17, -1e-300], k)
    y0[6 * k:7 * k] = tiny
    x0[6 * k:7 * k] = tiny * 3
    y1[6 * k:7 * k] = rng.uniform(0, 3, k)
    return x0, y0, x1, y1


@pytest.mark.parametrize("gt", [(0.0, 1.0, 0.0, 0.0, 0.0, 1.0), (1000.25, 0.3, 0.0, 2000.0, 0.0, -0.7),
                                (-5.0, -2.5, 0.0, 7.0, 0.0, 1.5)], ids=["identity", "south-down", "mirrored-x"])
def test_pixel_transform_is_numpys(core, gt):
    rng = np.random.default_rng(1)
    X = np.concatenate([rng.uniform(-1e4, 1e4, 5000), rng.normal(0, 1e200, 100), [0.0, -0.0, 1e-310, gt[0], gt[3]]])
    assert np.array_equal(bits(pixel(core, X, gt[0], gt[1])), bits((X - gt[0]) / gt[1]))
    assert np.array_equal(bits(pixel(core, X, gt[3], gt[5])), bits((X - gt[3]) / gt[5]))


@pytest.mark.parametrize("H,W", [(64, 48), (1, 7), (7, 1)])
def test_rows_crossings_and_columns_are_numpys(core, H, W):
    rng = np.random.default_rng(H * 100 + W)
    x0, y0, x1, y1 = segments(rng, 16000, H, W)
    # the predicate
    yc = np.arange(H, dtype=np.float64) + 0.5
    want = (y0[:, None] <= yc) != (y1[:, None] <= yc)                        # [segments, rows]
    got = np.empty(want.size, np.uint8)
    a0, a1, ac = (np.ascontiguousarray(np.broadcast_to(a, want.shape)).ravel() for a in (y0[:, None], y1[:, None], yc))
    core.crosses_host(D(a0.ctypes.data), D(a1.ctypes.data), D(ac.ctypes.data), ctypes.c_long(want.size),
                      D(got.ctypes.data))
    assert np.array_equal(got.reshape(want.shape).astype(bool), want)
    # the rows: exactly the rows in [0, H) the predicate holds for, as one run
    first, count = rows(core, y0, y1, H)
    r = np.arange(H)
    assert np.array_equal((r >= first[:, None]) & (r < (first + count)[:, None]), want)
    assert (count > 0).any() and (count == 0).any()
    # xi and its column on every crossing, with numpy's operation order
    s, rr = np.nonzero(want)
    yc_s = rr + 0.5
    with np.errstate(over="ignore", invalid="ignore"):                       # the huge segments overflow, as they do there
        want_xi = x0[s] + (yc_s - y0[s]) * (x1[s] - x0[s]) / (y1[s] - y0[s])
    got_xi = xi(core, x0[s], y0[s], x1[s], y1[s], yc_s)
    assert np.array_equal(bits(got_xi), bits(want_xi))
    fin = np.isfinite(want_xi)
    assert np.array_equal(col(core, want_xi[fin], W), np.clip(np.ceil(want_xi[fin] - 0.5), 0, W).astype(np.int64))


def test_column_ties_and_extremes(core):
    W = 10
    x = np.array([-1e300, -np.inf, -1.0, -0.0, 0.0, 0.5, 0.5000000000000001, 0.49999999999999994, 1.0, 4.5, 9.5, 10.0,
                  10.5, 10.6, 1e300, np.inf] + list(np.arange(-3, 14) + 0.5), np.float64)
    assert np.array_equal(col(core, x, W), np.clip(np.ceil(x - 0.5), 0, W).astype(np.int64))
    assert col(core, [np.nan], W)[0] == 0


# ---------------------------------------------------------------------------------------------------------------------
# read_polygon_rings
# ---------------------------------------------------------------------------------------------------------------------
def walk_records(path):
    """A record-by-record restatement of the .shp layout: list (per record) of lists of [k, 2] parts."""
    raw = open(path, "rb").read()
    out, off = [], 100
    while off + 8 <= len(raw):
        (clen,) = struct.unpack_from(">i", raw, off + 4)
        body = off + 8
        parts = []
        if struct.unpack_from("<i", raw, body)[0] in (5, 15, 25):
            n_parts, n_points = struct.unpack_from("<ii", raw, body + 36)
            starts = list(struct.unpack_from("<%di" % n_parts, raw, body + 44)) + [n_points]
            base = body + 44 + 4 * n_parts
            for i in range(n_parts):
                parts.append(np.array([struct.unpack_from("<dd", raw, base + 16 * j) for j in range(starts[i], starts[i + 1])],
                                      np.float64).reshape(-1, 2))
        out.append(parts)
        off = body + 2 * clen
    return out


def assert_rings_equal(rings, records):
    xy, off, rec, n = rings
    assert xy.dtype == np.float64 and off.dtype == np.int64 and rec.dtype == np.int32
    assert n == len(records) and len(off) == len(rec) + 1 and off[0] == 0 and off[-1] == len(xy)
    flat = [(r, p) for r, parts in enumerate(records) for p in parts]
    assert len(flat) == len(rec)
    for k, (r, p) in enumerate(flat):
        assert rec[k] == r and np.array_equal(xy[off[k]:off[k + 1]], p)


def scene(rng, n):
    polys = []
    for i in range(n):
        if i % 7 == 3:
            polys.append([])                                       # null record
            continue
        rings = []
        for _ in range(int(rng.integers(1, 4))):
            m = int(rng.integers(3, 12))
            ring = rng.uniform(-1e5, 1e5, (m, 2))
            rings.append(ring if i % 2 else np.concatenate([ring, ring[:1]]))
        polys.append(rings)
    return polys


def _patch_type(path, st):
    raw = bytearray(open(path, "rb").read())
    struct.pack_into("<i", raw, 32, st)
    off = 100
    while off < len(raw):
        (clen,) = struct.unpack_from(">i", raw, off + 4)
        if struct.unpack_from("<i", raw, off + 8)[0] != 0:
            struct.pack_into("<i", raw, off + 8, st)
        off += 8 + 2 * clen
    open(path, "wb").write(bytes(raw))


@pytest.mark.parametrize("shape_type", [5, 15, 25])
def test_read_polygon_rings_matches_read_polygons(tmp_path, shape_type):
    rng = np.random.default_rng(shape_type)
    path = str(tmp_path / "tile.shp")
    shapefile.write_polygon_shp(path, scene(rng, 60))
    if shape_type != 5:
        _patch_type(path, shape_type)        # the Z / M types keep X and Y where type 5 has them
    want = walk_records(path)
    rings = shapefile.read_polygon_rings(path)
    assert_rings_equal(rings, want)
    got = shapefile.read_polygons(path)
    assert len(got) == len(want) and all(len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))
                                         for a, b in zip(got, want))
    # without the .shx index the record headers are walked
    os.remove(path[:-4] + ".shx")
    assert_rings_equal(shapefile.read_polygon_rings(path), want)


def test_read_polygon_rings_edge_files(tmp_path):
    path = str(tmp_path / "e.shp")
    shapefile.write_polygon_shp(path, [[], []])                      # null records only
    xy, off, rec, n = shapefile.read_polygon_rings(path)
    assert n == 2 and xy.shape == (0, 2) and list(off) == [0] and len(rec) == 0
    assert shapefile.read_polygons(path) == [[], []]
    shapefile.write_point_shp(str(tmp_path / "p.shp"), [1.0], [2.0])
    with pytest.raises(ValueError, match="not a polygon"):
        shapefile.read_polygon_rings(str(tmp_path / "p.shp"))
    # a record whose first part does not start at its first point, and a file cut inside a record's points
    shapefile.write_polygon_shp(path, [[np.arange(8.0).reshape(4, 2)], [np.arange(6.0).reshape(3, 2)]])
    raw = bytearray(open(path, "rb").read())
    good = bytes(raw)
    struct.pack_into("<i", raw, 100 + 8 + 44, 1)
    open(path, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="corrupt"):
        shapefile.read_polygon_rings(path)
    open(path, "wb").write(good[:-8])
    with pytest.raises(ValueError, match="corrupt or truncated"):
        shapefile.read_polygon_rings(path)


# ---------------------------------------------------------------------------------------------------------------------
# the C ABI without CUDA
# ---------------------------------------------------------------------------------------------------------------------
def _call(L, H=4, W=4, ld=4, n_v=8, n_rings=2, n_records=2, cap=64, gt1=1.0, gt5=-1.0, ptr=16, ws_bytes=None,
          counts=16, labels=16, nodata=-1):
    ws = L.dm_rasterize_workspace_bytes(n_v, n_records, max(cap, 0)) if ws_bytes is None else ws_bytes
    return L.dm_rasterize(ptr, n_v, ptr, ptr, n_rings, n_records, 0.0, gt1, 0.0, gt5, None, nodata, H, W, ld, cap,
                          labels, counts, ptr, ws, None)


def test_abi_rejects_bad_arguments_before_any_work():
    """Every argument is checked before anything is enqueued: no CUDA call is made (the pointers are addresses nothing
    may dereference, so a CUDA call would fail first with DM_ERR_CUDA) and no kernel is launched."""
    from deepmerge_b200 import _lib
    L = _lib.lib()
    bad, short = _lib.DM_ERR_BAD_ARG, _lib.DM_ERR_WORKSPACE
    cases = {
        "negative H": dict(H=-1), "negative W": dict(W=-1), "ld < W": dict(ld=3),
        "2^32 vertex indices": dict(H=1 << 20, W=1 << 20, ld=1 << 20), "H >= 2^31": dict(H=1 << 31, W=1, ld=1),
        "capacity 2^31": dict(cap=1 << 31), "negative capacity": dict(cap=-1), "negative vertices": dict(n_v=-1),
        "negative rings": dict(n_rings=-1), "negative records": dict(n_records=-1), "records 2^31": dict(n_records=1 << 31),
        "gt1 = 0": dict(gt1=0.0), "gt5 = 0": dict(gt5=0.0), "null inputs": dict(ptr=None), "null counts": dict(counts=None),
        "null labels": dict(labels=None),
    }
    for name, kw in cases.items():
        n0 = L.dm_launch_count()
        assert _call(L, **kw) == bad, name
        assert L.dm_launch_count() == n0, name
    n0 = L.dm_launch_count()
    ws = L.dm_rasterize_workspace_bytes(8, 2, 64)
    assert _call(L, ws_bytes=ws - 1) == short
    assert L.dm_launch_count() == n0
    # the empty raster: nothing to do, and nothing to clear without counts
    assert _call(L, H=0, counts=None) == 0
    assert _call(L, W=0, ld=0, counts=None, ptr=None) == 0


def test_abi_workspace_query():
    from deepmerge_b200 import _lib
    L = _lib.lib()
    q = L.dm_rasterize_workspace_bytes
    assert q(-1, 1, 1) == 0 and q(1, -1, 1) == 0 and q(1, 1, -1) == 0 and q(1, 1, 1 << 31) == 0
    assert 0 < q(0, 0, 0) < q(1000, 10, 1000) < q(1000, 10, 100000)
    assert q(10 ** 6, 10, 1000) >= 8 * 10 ** 6              # per vertex: its crossing count and first key
    assert q(1000, 1 << 22, 1000) > q(1000, 10, 1000)        # the sort's per-record arrays
    assert q(1000, 10, 10 ** 6) >= 8 * 10 ** 6               # one u64 key per crossing


def test_python_argument_checks():
    import deepmerge_b200 as dm
    sq = [[np.array([[0, 0], [1, 0], [1, 1]], float)]]
    with pytest.raises(ValueError, match="north-up"):
        dm.rasterize(sq, (0, 1, 0.5, 0, 0, -1), 4, 4)
    with pytest.raises(ValueError, match="north-up"):
        dm.rasterize(sq, (0, 0, 0, 0, 0, -1), 4, 4)
    with pytest.raises(ValueError, match="nodata"):
        dm.rasterize(sq, (0, 1, 0, 0, 0, -1), 4, 4, nodata=1 << 31)
    with pytest.raises(ValueError, match="CUDA"):
        dm.rasterize(sq, (0, 1, 0, 0, 0, -1), 4, 4, device="cpu")
