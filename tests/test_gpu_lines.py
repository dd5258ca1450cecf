"""GPU: dm_lines bit for bit against the sequential tracer of tests/lines_oracle.c (dmo_lines), on the rasters of
test_lines_cpu, on synthetic Voronoi scenes before and after merging, on odd sizes and strided views, end to end
through the reference's scoring of lines.shp, and on the configs[1] scene at full size (10k x 10k)."""
import numpy as np
import pytest

import lines_oracle as lo
from oracle import oracle_np as o
from test_lines_cpu import CASES, check_invariants

pytestmark = pytest.mark.gpu

FIELDS = ("line_left", "line_right", "line_length", "line_offsets", "vertices")


def gpu(P):
    return {f: getattr(P, f).cpu().numpy() for f in FIELDS}


def assert_same(P, want):
    got = gpu(P)
    for f in FIELDS:
        assert np.array_equal(got[f], want[f]), f
    assert P.boundary_segments == want["counts"][2]


def run(cuda, L, R, **kw):
    import torch
    from deepmerge_b200 import boundary_lines
    return boundary_lines(torch.from_numpy(np.ascontiguousarray(L)).to(cuda), R, **kw)


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_oracle_on_cpu_cases(cuda, name):
    L, R = CASES[name]
    assert_same(run(cuda, L, R), lo.lines(L, R))


@pytest.mark.parametrize("H,W", [(1024, 1024), (333, 517), (97, 45)])
def test_matches_oracle_on_voronoi_unmerged_and_merged(cuda, H, W):
    import torch
    from deepmerge_b200 import merge_scene
    sc = o.synth_scene(H, W, 2000 * H * W // (1024 * 1024) + 8, C=4)
    L, R = sc["labels"], sc["n_regions"]
    assert_same(run(cuda, L, R), lo.lines(L, R))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    res = merge_scene(t(L), t(sc["feats"]), 0.5, n_regions=R, image=t(sc["image"]), xs=t(sc["xs"]), ys=t(sc["ys"]))
    M = res.labels.cpu().numpy()
    want = lo.lines(M, R)
    assert_same(run(cuda, M, R), want)
    check_invariants(M, R, want)


def test_strided_view(cuda):
    import torch
    from deepmerge_b200 import boundary_lines
    L, R = o.synth_labels(200, 300, 500, seed=5)
    L = L.copy()
    L[50:60, 70:90] = -1
    big = torch.full((200, 333), 7, dtype=torch.int32, device=cuda)
    big[:, 13:313] = torch.from_numpy(L).to(cuda)
    view = big[:, 13:313]
    assert view.stride(0) == 333
    assert_same(boundary_lines(view, R), lo.lines(L, R))


def test_capacity_retry_and_status(cuda):
    import torch
    from deepmerge_b200 import _lib, boundary_lines
    L, R = o.synth_labels(128, 160, 200, seed=9)
    want = lo.lines(L, R)
    segs = int(want["counts"][2])
    assert_same(boundary_lines(torch.from_numpy(L).to(cuda), R, capacity=64), want)
    # the raw ABI: a small capacity reports status 2 and the exact segment count; an exact one succeeds
    lib = _lib.lib()
    lab = torch.from_numpy(L).to(cuda)
    stream = torch.cuda.current_stream().cuda_stream
    for cap, status in ((64, 2), (segs, 0)):
        ws_bytes = lib.dm_lines_workspace_bytes(128, 160, cap)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda)
        bufs = [torch.empty(cap, dtype=torch.int32, device=cuda), torch.empty(cap, dtype=torch.int32, device=cuda),
                torch.empty(cap, dtype=torch.int64, device=cuda), torch.empty(cap + 1, dtype=torch.int64, device=cuda),
                torch.empty((2 * cap, 2), dtype=torch.int32, device=cuda)]
        counts = torch.zeros(4, dtype=torch.int64, device=cuda)
        rc = lib.dm_lines(lab.data_ptr(), 128, 160, 160, R, cap, *[b.data_ptr() for b in bufs], counts.data_ptr(),
                          ws.data_ptr(), ws_bytes, stream)
        assert rc == 0
        c = counts.tolist()
        assert c[3] == status and c[2] == segs
        if status == 0:
            assert c[0] == len(want["line_left"]) and c[1] == len(want["vertices"])
            assert np.array_equal(bufs[4][:c[1]].cpu().numpy(), want["vertices"])


def test_label_out_of_range_raises(cuda):
    L = np.zeros((40, 50), np.int32)
    L[10, 20] = 3
    with pytest.raises(ValueError):
        run(cuda, L, 3)


def test_two_calls_are_bit_equal(cuda):
    L, R = o.synth_labels(512, 384, 900, seed=2)
    a, b = gpu(run(cuda, L, R)), gpu(run(cuda, L, R))
    for f in FIELDS:
        assert np.array_equal(a[f], b[f])


def test_workspace_fits_the_queried_size(cuda):
    """Everything the call touches in its workspace lies inside the queried size: the bytes after it keep a sentinel."""
    import torch
    from deepmerge_b200 import _lib
    lib = _lib.lib()
    L, R = o.synth_labels(300, 200, 400, seed=6)
    want = lo.lines(L, R)
    cap = int(want["counts"][2]) + 100
    ws_bytes = lib.dm_lines_workspace_bytes(300, 200, cap)
    ws = torch.full((ws_bytes + 4096,), 0x5A, dtype=torch.uint8, device=cuda)
    bufs = [torch.empty(cap, dtype=torch.int32, device=cuda), torch.empty(cap, dtype=torch.int32, device=cuda),
            torch.empty(cap, dtype=torch.int64, device=cuda), torch.empty(cap + 1, dtype=torch.int64, device=cuda),
            torch.empty((2 * cap, 2), dtype=torch.int32, device=cuda)]
    counts = torch.zeros(4, dtype=torch.int64, device=cuda)
    lab = torch.from_numpy(L).to(cuda)
    assert lib.dm_lines(lab.data_ptr(), 300, 200, 200, R, cap, *[b.data_ptr() for b in bufs], counts.data_ptr(),
                        ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream) == 0
    c = counts.tolist()
    assert c[3] == 0 and c[0] == len(want["line_left"])
    assert (ws[ws_bytes:] == 0x5A).all()
    assert np.array_equal(bufs[2][:c[0]].cpu().numpy(), want["line_length"])


def test_end_to_end_through_the_reference_scoring(cuda, tmp_path):
    """polygons on disk -> rasterize -> write_polygonized (tile.shp, + PointID) and write_boundary_lines (lines.shp)
    -> the reference's test_for_shp: every simi is the distance of the two polygons' mean rows, and the edge list the
    reference's reader takes from lines.shp is the RAG of the raster."""
    import torch
    from deepmerge_b200 import boundary_lines, polygonize
    from deepmerge_b200 import shapefile as shp
    from deepmerge_b200.ExtractFeatures import test_for_shp
    from deepmerge_b200.MyUtils2 import PolygonConnectPointDataset
    rng = np.random.default_rng(4)
    H, W = 120, 160
    gt = (1000.0, 0.5, 0.0, 2000.0, 0.0, -0.5)
    polys = []
    for i in range(60):
        x0, y0 = rng.uniform(0, W - 10), rng.uniform(0, H - 10)
        w, h = rng.uniform(4, 40), rng.uniform(4, 30)
        pix = np.array([[x0, y0], [x0 + w, y0], [x0 + w, y0 + h], [x0, y0 + h]])
        polys.append([np.stack([gt[0] + pix[:, 0] * gt[1], gt[3] + pix[:, 1] * gt[5]], 1)])
    src = str(tmp_path / "source.shp")
    shp.write_polygon_shp(src, polys)
    labels = shp.rasterize_polygons(shp.read_polygons(src), gt, H, W)
    R = len(polys)
    lab = torch.from_numpy(labels).to(cuda)
    tile, lines_path = str(tmp_path / "tile.shp"), str(tmp_path / "lines.shp")
    shp.write_polygonized(tile, polygonize(lab, R), gt)
    shp.write_boundary_lines(lines_path, boundary_lines(lab, R), gt)
    # sample points: every pixel centre of every tenth row / column that is not nodata, PointID lists per record
    ys, xs = np.nonzero(labels >= 0)
    keep = (ys % 10 == 3) & (xs % 10 == 7)
    ys, xs = ys[keep], xs[keep]
    points = str(tmp_path / "points.shp")
    shp.write_point_shp(points, gt[0] + (xs + 0.5) * gt[1], gt[3] + (ys + 0.5) * gt[5])
    shp.write_dbf(points[:-4] + ".dbf", [shp.FieldDefn("ID", "N", 9, 0)], {"ID": list(range(len(xs)))})
    region = shp.DbfTable(tile[:-4] + ".dbf").column_int("REGION")
    store = rng.standard_normal((len(xs), 16)).astype(np.float32)
    rec_of_point = np.searchsorted(region, labels[ys, xs])
    pid = [" ".join(str(i) for i in np.flatnonzero(rec_of_point == r)) for r in range(len(region))]
    t = shp.DbfTable(tile[:-4] + ".dbf", update=True)
    t.add_field(shp.FieldDefn("PointID", "C", 254))
    t.set_column("PointID", pid)
    t.flush()
    assert test_for_shp(store, None, tile, lines_path, points) == 0
    lt = shp.DbfTable(lines_path[:-4] + ".dbf")
    lf, rf, simi = lt.column_int("LEFT_FID"), lt.column_int("RIGHT_FID"), lt.column_float("simi")
    means = np.stack([store[rec_of_point == r].mean(0) if (rec_of_point == r).any() else np.full(16, np.nan, np.float32)
                      for r in range(len(region))]).astype(np.float64)
    both = (lf >= 0) & (rf >= 0)
    assert both.any() and np.isnan(simi[~both]).all()
    want = np.linalg.norm(means[lf[both]] - means[rf[both]], axis=1)
    ok = ~np.isnan(want)
    assert ok.any() and np.allclose(simi[both][ok], want[ok], rtol=1e-5, atol=1e-5)
    ds = PolygonConnectPointDataset(None, tile, lines_path, points)
    k = ds.edge_keys()
    a, b = region[k >> 32], region[k & 0xFFFFFFFF]
    got = set(((np.minimum(a, b) << 32) | np.maximum(a, b)).tolist())
    assert got == set(o.build_rag(labels, R)[0].astype(np.int64).tolist())


def test_configs1_full_size_merged(cuda):
    """configs[1] (10k x 10k, ~100k regions): the merged map of MergeEngine.run, bit-exact against the oracle, and the
    boundary-length / perimeter identities against the merge's own statistics."""
    import torch
    from deepmerge_b200 import MergeEngine, boundary_lines
    from deepmerge_b200.synth import synth_scene
    H = W = 10000
    sc = synth_scene(H, W, 100000, C=4, device=cuda)
    eng = MergeEngine(H, W, sc.n_regions, sc.feats.shape[1], C=4, n_points=sc.feats.shape[0], device=cuda)
    res = eng.run(sc.labels, sc.feats, 0.5, image=sc.image, xs=sc.xs, ys=sc.ys)
    P = boundary_lines(res.labels, sc.n_regions)
    M = res.labels.cpu().numpy()
    assert_same(P, lo.lines(M, sc.n_regions))
    R = sc.n_regions
    lf, rt, ln = (t.cpu().numpy().astype(np.int64) for t in (P.line_left, P.line_right, P.line_length))
    both = lf >= 0
    keys, inv = np.unique((lf[both] << 32) | rt[both], return_inverse=True)
    blen = np.bincount(inv, weights=ln[both]).astype(np.int64)
    assert np.array_equal(keys, res.edge_keys.cpu().numpy().astype(np.int64))
    assert np.array_equal(blen, res.boundary_len.cpu().numpy().astype(np.int64))
    per = np.zeros(R, np.int64)
    np.add.at(per, rt, ln)
    np.add.at(per, lf[both], ln[both])
    roots = (res.root == torch.arange(R, device=cuda, dtype=torch.int32)).cpu().numpy()
    assert np.array_equal(per[roots], res.perimeter.cpu().numpy()[roots])
