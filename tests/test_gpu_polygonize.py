"""GPU: dm_polygonize bit for bit against the sequential tracer of tests/polygon_oracle.c (dmo_polygonize), on the
hand-made and random rasters of test_polygonize_cpu, on synthetic Voronoi scenes before and after merging, on odd sizes
and strided views, and on the configs[1] scene at full size (10k x 10k)."""
import numpy as np
import pytest

import polygon_oracle as po
from oracle import oracle_np as o
from test_polygonize_cpu import CASES, check_invariants, check_round_trip

pytestmark = pytest.mark.gpu

FIELDS = ("ring_region", "ring_offsets", "ring_area", "vertices", "region_rings")


def gpu(P):
    return {f: getattr(P, f).cpu().numpy() for f in FIELDS}


def assert_same(P, want):
    got = gpu(P)
    for f in FIELDS:
        assert np.array_equal(got[f], want[f]), f
    assert P.boundary_sides == want["counts"][2]


def run(cuda, L, R, **kw):
    import torch
    from deepmerge_b200 import polygonize
    return polygonize(torch.from_numpy(np.ascontiguousarray(L)).to(cuda), R, **kw)


@pytest.mark.parametrize("name", sorted(CASES))
def test_matches_oracle_on_cpu_cases(cuda, name):
    L, R = CASES[name]
    assert_same(run(cuda, L, R), po.polygonize(L, R))


@pytest.mark.parametrize("H,W", [(1024, 1024), (333, 517), (97, 45)])
def test_matches_oracle_on_voronoi_unmerged_and_merged(cuda, H, W):
    import torch
    from deepmerge_b200 import merge_scene
    sc = o.synth_scene(H, W, 2000 * H * W // (1024 * 1024) + 8, C=4)
    L, R = sc["labels"], sc["n_regions"]
    assert_same(run(cuda, L, R), po.polygonize(L, R))
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    res = merge_scene(t(L), t(sc["feats"]), 0.5, n_regions=R, image=t(sc["image"]), xs=t(sc["xs"]), ys=t(sc["ys"]))
    M = res.labels.cpu().numpy()
    P = run(cuda, M, R)
    want = po.polygonize(M, R)
    assert_same(P, want)
    check_invariants(M, R, want)
    roots = (res.root == torch.arange(R, device=cuda, dtype=torch.int32)).cpu().numpy()
    assert np.array_equal(P.region_area(R).cpu().numpy()[roots], res.area.cpu().numpy()[roots])


def test_strided_view(cuda):
    import torch
    from deepmerge_b200 import polygonize
    L, R = o.synth_labels(200, 300, 500, seed=5)
    L = L.copy()
    L[50:60, 70:90] = -1
    big = torch.full((200, 333), 7, dtype=torch.int32, device=cuda)
    big[:, 13:313] = torch.from_numpy(L).to(cuda)
    view = big[:, 13:313]
    assert view.stride(0) == 333
    assert_same(polygonize(view, R), po.polygonize(L, R))


def test_capacity_retry_and_status(cuda):
    import torch
    from deepmerge_b200 import _lib, polygonize
    L, R = o.synth_labels(128, 160, 200, seed=9)
    want = po.polygonize(L, R)
    sides = int(want["counts"][2])
    assert_same(polygonize(torch.from_numpy(L).to(cuda), R, capacity=64), want)
    # the raw ABI: a small capacity reports status 2 and the exact side count
    lib = _lib.lib()
    lab = torch.from_numpy(L).to(cuda)
    cap = 64
    ws_bytes = lib.dm_polygonize_workspace_bytes(128, 160, R, cap)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda)
    bufs = [torch.empty(cap // 4, dtype=torch.int32, device=cuda), torch.empty(cap // 4 + 1, dtype=torch.int64, device=cuda),
            torch.empty(cap // 4, dtype=torch.int64, device=cuda), torch.empty((cap, 2), dtype=torch.int32, device=cuda),
            torch.empty(R + 1, dtype=torch.int64, device=cuda)]
    counts = torch.zeros(4, dtype=torch.int64, device=cuda)
    rc = lib.dm_polygonize(lab.data_ptr(), 128, 160, 160, R, cap, *[b.data_ptr() for b in bufs], counts.data_ptr(),
                           ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    c = counts.tolist()
    assert c[3] == 2 and c[2] == sides


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


def test_end_to_end_from_files(cuda, tmp_path):
    """polygons on disk -> rasterize -> merge -> polygonize -> write -> read -> rasterize == the merged labels"""
    import torch
    from deepmerge_b200 import merge_scene, polygonize
    from deepmerge_b200 import shapefile as shp
    rng = np.random.default_rng(4)
    H, W = 120, 160
    gt = (1000.0, 0.5, 0.0, 2000.0, 0.0, -0.5)
    polys = []
    for i in range(60):
        x0, y0 = rng.uniform(0, W - 10), rng.uniform(0, H - 10)
        w, h = rng.uniform(4, 40), rng.uniform(4, 30)
        if i % 3 == 0:       # a random star-shaped polygon
            ang = np.sort(rng.uniform(0, 2 * np.pi, 7))
            rad = rng.uniform(3, 15, 7)
            pix = np.stack([x0 + rad * np.cos(ang), y0 + rad * np.sin(ang)], 1)
        else:
            pix = np.array([[x0, y0], [x0 + w, y0], [x0 + w, y0 + h], [x0, y0 + h]])
        polys.append([np.stack([gt[0] + pix[:, 0] * gt[1], gt[3] + pix[:, 1] * gt[5]], 1)])
    src = str(tmp_path / "tile.shp")
    shp.write_polygon_shp(src, polys)
    labels = shp.rasterize_polygons(shp.read_polygons(src), gt, H, W)
    R = len(polys)
    ys, xs = np.nonzero(labels >= 0)
    pick = rng.choice(len(xs), 400, replace=False)
    xs, ys = xs[pick].astype(np.int32), ys[pick].astype(np.int32)
    feats = (labels[ys, xs] % 5).astype(np.float32)[:, None] * np.ones((1, 8), np.float32)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    res = merge_scene(t(labels), t(feats), 0.5, n_regions=R, xs=t(xs), ys=t(ys))
    M = res.labels.cpu().numpy()
    P = polygonize(res.labels, R)
    want = po.polygonize(M, R)
    assert_same(P, want)
    check_round_trip(M, want, tmp_path, columns={"PERI": res.perimeter.cpu().numpy()})
    out = str(tmp_path / "tile_merged.shp")
    shp.write_polygonized(out, P, gt, {"PERI": res.perimeter})
    ids = shp.DbfTable(out[:-4] + ".dbf").column_int("REGION")
    assert np.array_equal(shp.rasterize_polygons(shp.read_polygons(out), gt, H, W, ids=ids), M)


def test_configs1_full_size_merged(cuda):
    """configs[1] (10k x 10k, ~100k regions): the merged map of MergeEngine.run, bit-exact against the oracle, and the
    area / perimeter identities against the merge's own statistics."""
    import torch
    from deepmerge_b200 import MergeEngine
    from deepmerge_b200.synth import synth_scene
    H = W = 10000
    sc = synth_scene(H, W, 100000, C=4, device=cuda)
    eng = MergeEngine(H, W, sc.n_regions, sc.feats.shape[1], C=4, n_points=sc.feats.shape[0], device=cuda)
    res = eng.run(sc.labels, sc.feats, 0.5, image=sc.image, xs=sc.xs, ys=sc.ys)
    from deepmerge_b200 import polygonize
    P = polygonize(res.labels, sc.n_regions)
    M = res.labels.cpu().numpy()
    assert_same(P, po.polygonize(M, sc.n_regions))
    R = sc.n_regions
    roots = (res.root == torch.arange(R, device=cuda, dtype=torch.int32)).cpu().numpy()
    assert np.array_equal(P.region_area(R).cpu().numpy()[roots], res.area.cpu().numpy()[roots])
    v = P.vertices.cpu().numpy().astype(np.int64)
    off = P.ring_offsets.cpu().numpy()
    rr = P.ring_region.cpu().numpy()
    d = np.abs(np.roll(v, -1, axis=0) - v).sum(1)
    last = off[1:] - 1                                        # closing edge of every ring: back to its first vertex
    d[last] = np.abs(v[last] - v[off[:-1]]).sum(1)
    per = np.zeros(R, np.int64)
    np.add.at(per, np.repeat(rr, np.diff(off)), d)
    assert np.array_equal(per[roots], res.perimeter.cpu().numpy()[roots])
