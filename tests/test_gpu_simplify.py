"""GPU: dm_polygonize_simplified and dm_lines_simplified bit for bit against the sequential simplifier of
tests/simplify_oracle.c, on the rasters of test_simplify_cpu, on synthetic Voronoi scenes before and after merging, on
strided views and on the configs[1] scene at full size (10k x 10k), where the shared-boundary and area identities are
checked on the GPU's output; end to end through the shapefile writers and readers."""
import numpy as np
import pytest

import simplify_oracle as so
from oracle import oracle_np as o
from test_simplify_cpu import CASES, TOLERANCES

pytestmark = pytest.mark.gpu

POLY_FIELDS = ("ring_region", "ring_offsets", "ring_area", "vertices", "region_rings")
LINE_FIELDS = ("line_left", "line_right", "line_length", "line_offsets", "vertices")


def host(P, fields):
    return {f: getattr(P, f).cpu().numpy() for f in fields}


def assert_same(P, want, fields):
    got = host(P, fields)
    for f in fields:
        assert np.array_equal(got[f], want[f]), f


def both(cuda, L, R, t, **kw):
    """(polygonize, boundary_lines) at tolerance t on the GPU"""
    import torch
    from deepmerge_b200 import boundary_lines, polygonize
    lab = L if isinstance(L, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(L)).to(cuda)
    return polygonize(lab, R, tolerance=t, **kw), boundary_lines(lab, R, tolerance=t, **kw)


def check_against_oracle(cuda, L, R, tolerances=TOLERANCES):
    for t in tolerances:
        P, Q = both(cuda, L, R, t)
        assert_same(P, so.polygons(L, R, t), POLY_FIELDS)
        assert_same(Q, so.lines(L, R, t), LINE_FIELDS)


def _next_in_chain(off, n, cyclic):
    """index of the vertex after each vertex of its chain (cyclic: wrapping), -1 after the last of a line"""
    nxt = np.arange(1, n + 1, dtype=np.int64)
    ends = off[1:] - 1
    nxt[ends] = off[:-1] if cyclic else -1
    return nxt


def check_shared_boundaries(P, Q, H, W, nodata):
    """Every directed edge of a simplified ring, tagged with its region, is an edge of a simplified line: forward for
    line_right, reversed for line_left (both multisets are equal).  Without nodata the doubled ring areas sum to 2 H W."""
    rv = P.vertices.cpu().numpy().astype(np.int64)
    roff = P.ring_offsets.cpu().numpy()
    reg = np.repeat(P.ring_region.cpu().numpy().astype(np.int64), np.diff(roff))
    key = lambda v: v[:, 1] * (W + 1) + v[:, 0]       # noqa: E731
    rk = key(rv)
    rn = _next_in_chain(roff, len(rv), True)
    ring_edges = np.stack([reg, rk, rk[rn]], 1)
    lv = Q.vertices.cpu().numpy().astype(np.int64)
    loff = Q.line_offsets.cpu().numpy()
    lk = key(lv)
    ln = _next_in_chain(loff, len(lv), False)
    has = ln >= 0
    left = np.repeat(Q.line_left.cpu().numpy().astype(np.int64), np.diff(loff))[has]
    right = np.repeat(Q.line_right.cpu().numpy().astype(np.int64), np.diff(loff))[has]
    a, b = lk[has], lk[ln[has]]
    fwd = np.stack([right, a, b], 1)
    rev = np.stack([left, b, a], 1)[left >= 0]
    line_edges = np.concatenate([fwd, rev])
    srt = lambda e: e[np.lexsort(e.T[::-1])]           # noqa: E731
    assert np.array_equal(srt(ring_edges), srt(line_edges)), "a ring and a line disagree on a shared boundary"
    if not nodata:
        x, y = rv[:, 0], rv[:, 1]
        assert int((x * y[rn] - x[rn] * y).sum()) == 2 * H * W


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_oracle_on_cpu_cases(cuda, name):
    L, R = CASES[name]
    check_against_oracle(cuda, L, R)
    if L.size:
        P, Q = both(cuda, L, R, 1.0)
        check_shared_boundaries(P, Q, *L.shape, nodata=bool((L < 0).any()))


@pytest.mark.parametrize("H,W", [(1024, 1024), (333, 517), (97, 45)])
def test_matches_oracle_on_voronoi_unmerged_and_merged(cuda, H, W):
    import torch
    from deepmerge_b200 import merge_scene
    sc = o.synth_scene(H, W, 2000 * H * W // (1024 * 1024) + 8, C=4)
    L, R = sc["labels"], sc["n_regions"]
    check_against_oracle(cuda, L, R)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)     # noqa: E731
    res = merge_scene(t(L), t(sc["feats"]), 0.5, n_regions=R, image=t(sc["image"]), xs=t(sc["xs"]), ys=t(sc["ys"]))
    M = res.labels.cpu().numpy()
    check_against_oracle(cuda, M, R)
    P, Q = both(cuda, M, R, 1.5)
    check_shared_boundaries(P, Q, H, W, nodata=False)


def test_strided_view(cuda):
    import torch
    L, R = o.synth_labels(200, 300, 500, seed=5)
    L = L.copy()
    L[50:60, 70:90] = -1
    big = torch.full((200, 333), 7, dtype=torch.int32, device=cuda)
    big[:, 13:313] = torch.from_numpy(L).to(cuda)
    view = big[:, 13:313]
    assert view.stride(0) == 333
    for t in (0.5, 4.0):
        P, Q = both(cuda, view, R, t)
        assert_same(P, so.polygons(L, R, t), POLY_FIELDS)
        assert_same(Q, so.lines(L, R, t), LINE_FIELDS)


def test_capacity_retry_and_two_calls(cuda):
    L, R = o.synth_labels(128, 160, 200, seed=9)
    P, Q = both(cuda, L, R, 1.0, capacity=64)
    assert_same(P, so.polygons(L, R, 1.0), POLY_FIELDS)
    assert_same(Q, so.lines(L, R, 1.0), LINE_FIELDS)
    P2, Q2 = both(cuda, L, R, 1.0)
    assert_same(P2, host(P, POLY_FIELDS), POLY_FIELDS)
    assert_same(Q2, host(Q, LINE_FIELDS), LINE_FIELDS)


def test_label_out_of_range_raises(cuda):
    import torch
    from deepmerge_b200 import boundary_lines, polygonize
    L = torch.zeros((40, 50), dtype=torch.int32, device=cuda)
    L[10, 20] = 3
    for f in (polygonize, boundary_lines):
        with pytest.raises(ValueError):
            f(L, 3, tolerance=1.0)


def test_bad_tolerance_raises(cuda):
    L = np.zeros((4, 5), np.int32)
    for t in (float("nan"), float("inf"), -0.5):
        with pytest.raises(ValueError):
            both(cuda, L, 1, t)


def test_workspace_fits_the_queried_size(cuda):
    """Everything each call touches in its workspace lies inside the queried size: the bytes after it keep a sentinel."""
    import torch
    from deepmerge_b200 import _lib
    lib = _lib.lib()
    L, R = o.synth_labels(300, 200, 400, seed=6)
    H, W = L.shape
    lab = torch.from_numpy(L).to(cuda)
    stream = torch.cuda.current_stream().cuda_stream
    dev = dict(device=cuda)
    # polygons
    want = so.polygons(L, R, 1.0)
    cap = int(want["counts"][2]) + 100
    rc = cap // 4
    ws_bytes = lib.dm_polygonize_simplified_workspace_bytes(H, W, R, cap)
    ws = torch.full((ws_bytes + 4096,), 0x5A, dtype=torch.uint8, **dev)
    bufs = [torch.empty(rc, dtype=torch.int32, **dev), torch.empty(rc + 1, dtype=torch.int64, **dev),
            torch.empty(rc, dtype=torch.int64, **dev), torch.empty((cap, 2), dtype=torch.int32, **dev),
            torch.empty(R + 1, dtype=torch.int64, **dev)]
    counts = torch.zeros(4, dtype=torch.int64, **dev)
    assert lib.dm_polygonize_simplified(lab.data_ptr(), H, W, W, R, cap, 1.0, *[b.data_ptr() for b in bufs],
                                        counts.data_ptr(), ws.data_ptr(), ws_bytes, stream) == 0
    c = counts.tolist()
    assert c[3] == 0 and c[1] == len(want["vertices"])
    assert (ws[ws_bytes:] == 0x5A).all()
    assert np.array_equal(bufs[3][:c[1]].cpu().numpy(), want["vertices"])
    # lines
    want = so.lines(L, R, 1.0)
    cap = int(want["counts"][2]) + 100
    ws_bytes = lib.dm_lines_simplified_workspace_bytes(H, W, cap)
    ws = torch.full((ws_bytes + 4096,), 0x5A, dtype=torch.uint8, **dev)
    bufs = [torch.empty(cap, dtype=torch.int32, **dev), torch.empty(cap, dtype=torch.int32, **dev),
            torch.empty(cap, dtype=torch.int64, **dev), torch.empty(cap + 1, dtype=torch.int64, **dev),
            torch.empty((2 * cap, 2), dtype=torch.int32, **dev)]
    counts = torch.zeros(4, dtype=torch.int64, **dev)
    assert lib.dm_lines_simplified(lab.data_ptr(), H, W, W, R, cap, 1.0, *[b.data_ptr() for b in bufs],
                                   counts.data_ptr(), ws.data_ptr(), ws_bytes, stream) == 0
    c = counts.tolist()
    assert c[3] == 0 and c[1] == len(want["vertices"])
    assert (ws[ws_bytes:] == 0x5A).all()
    assert np.array_equal(bufs[4][:c[1]].cpu().numpy(), want["vertices"])


def test_end_to_end_through_the_shapefiles(cuda, tmp_path):
    """write_polygonized / write_boundary_lines of simplified outputs: the geometry read back is the outputs', and
    LEFT_FID / RIGHT_FID are still the record indices of the polygon file."""
    import torch
    from deepmerge_b200 import boundary_lines, polygonize
    from deepmerge_b200 import shapefile as shp
    L, R = o.synth_labels(150, 210, 120, seed=12)
    L = L.copy()
    L[20:30, 40:70] = -1
    gt = (500.0, 2.0, 0.0, 900.0, 0.0, -2.0)
    lab = torch.from_numpy(L).to(cuda)
    P, Q = polygonize(lab, R, tolerance=1.5), boundary_lines(lab, R, tolerance=1.5)
    tile, lines_path = str(tmp_path / "tile.shp"), str(tmp_path / "lines.shp")
    shp.write_polygonized(tile, P, gt)
    shp.write_boundary_lines(lines_path, Q, gt)
    ids, rings = P.shapes(gt)
    back = shp.read_polygons(tile)
    assert len(back) == len(rings)
    for got, want in zip(back, rings):
        assert len(got) == len(want) and all(np.array_equal(np.asarray(g), w) for g, w in zip(got, want))
    lines = shp.read_polylines(lines_path)
    want = Q.shapes(gt)
    assert len(lines) == len(want)
    for got, w in zip(lines, want):
        assert len(got) == 1 and np.array_equal(np.asarray(got[0]), w)
    region = shp.DbfTable(tile[:-4] + ".dbf").column_int("REGION")
    lt = shp.DbfTable(lines_path[:-4] + ".dbf")
    lf, rf = lt.column_int("LEFT_FID"), lt.column_int("RIGHT_FID")
    left, right = Q.line_left.cpu().numpy(), Q.line_right.cpu().numpy()
    assert np.array_equal(region[rf], right)
    assert np.array_equal(np.where(lf >= 0, region[np.maximum(lf, 0)], -1), left)
    assert np.array_equal(shp.DbfTable(tile[:-4] + ".dbf").column_int("AREA"), np.bincount(L[L >= 0])[region])


@pytest.fixture(scope="module")
def configs1(cuda):
    """configs[1] (10k x 10k, ~100k regions): the unmerged synthetic labels and the merged map of MergeEngine.run"""
    from deepmerge_b200 import MergeEngine
    from deepmerge_b200.synth import synth_scene
    H = W = 10000
    sc = synth_scene(H, W, 100000, C=4, device=cuda)
    eng = MergeEngine(H, W, sc.n_regions, sc.feats.shape[1], C=4, n_points=sc.feats.shape[0], device=cuda)
    res = eng.run(sc.labels, sc.feats, 0.5, image=sc.image, xs=sc.xs, ys=sc.ys)
    return {"unmerged": sc.labels, "merged": res.labels.clone()}, sc.n_regions


@pytest.mark.parametrize("which", ["merged", "unmerged"])
def test_configs1_full_size(cuda, configs1, which):
    maps, R = configs1
    lab = maps[which]
    P, Q = both(cuda, lab, R, 1.0)
    M = lab.cpu().numpy()
    assert_same(P, so.polygons(M, R, 1.0), POLY_FIELDS)
    assert_same(Q, so.lines(M, R, 1.0), LINE_FIELDS)
    check_shared_boundaries(P, Q, *M.shape, nodata=bool((M < 0).any()))
