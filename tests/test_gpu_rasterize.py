"""GPU: deepmerge_b200.rasterize (dm_rasterize) bit for bit against shapefile.rasterize_polygons, on hand-made and seeded
random scenes (overlaps, bow-ties, vertices on pixel centres and corners, rings outside the raster, closed and unclosed
rings, rings of fewer than 3 vertices, empty records, ids and nodata, three geotransforms), on a polygon with more
crossings than the sort's bucket limit, on thousands of tiny polygons and on odd sizes; the raw ABI's strided output,
capacity status and error statuses; and the round trips label raster -> polygonize -> rasterize, in memory (configs[1]
at full size included) and through the shapefile writer and the flat reader."""
import numpy as np
import pytest

from deepmerge_b200 import shapefile as shp
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu

IDENTITY = (0.0, 1.0, 0.0, 0.0, 0.0, 1.0)
TRANSFORMS = {"north-up": (1000.0, 0.5, 0.0, 2000.0, 0.0, -0.5), "south-down": (1000.25, 0.3, 0.0, 2000.0, 0.0, 0.7),
              "mirrored-x": (-5.0, -2.5, 0.0, 7.0, 0.0, -1.5)}


def gpu(polys, gt, H, W, **kw):
    import torch
    import deepmerge_b200 as dm
    out = dm.rasterize(polys, gt, H, W, **kw)
    assert out.is_cuda and out.dtype == torch.int32 and tuple(out.shape) == (H, W)
    return out.cpu().numpy()


def assert_matches(polys, gt, H, W, **kw):
    want = shp.rasterize_polygons(polys, gt, H, W, **kw)
    got = gpu(polys, gt, H, W, **kw)
    assert np.array_equal(got, want), int((got != want).sum())
    return got


def to_map(pix, gt):
    return np.stack([gt[0] + pix[:, 0] * gt[1], gt[3] + pix[:, 1] * gt[5]], 1)


def crossings(polys, gt, H):
    """The number of (segment, row) crossings, from the rules of rasterize_polygons."""
    n = 0
    yc = np.arange(H) + 0.5
    for rings in polys:
        for r in rings:
            r = np.asarray(r, np.float64).reshape(-1, 2)
            if len(r) < 3:
                continue
            px, py = (r[:, 0] - gt[0]) / gt[1], (r[:, 1] - gt[3]) / gt[5]
            if px[0] != px[-1] or py[0] != py[-1]:
                py = np.append(py, py[0])
            n += int(((py[:-1, None] <= yc) != (py[1:, None] <= yc)).sum())
    return n


def random_scene(rng, H, W, gt, n):
    """n records in map coordinates: stars, bow-ties, vertices snapped to pixel centres and corners, rings partly or
    wholly outside the raster, rings of 1-2 vertices, empty records; every other ring explicitly closed."""
    polys = []
    for _ in range(n):
        kind = int(rng.integers(0, 7))
        if kind == 0:
            polys.append([])
            continue
        rings = []
        for _ in range(int(rng.integers(1, 4))):
            cx, cy = rng.uniform(-0.2 * W, 1.2 * W), rng.uniform(-0.2 * H, 1.2 * H)
            m = int(rng.integers(1, 12))
            if kind == 1:                                        # pixel centres and corners
                pix = np.stack([np.round(cx + rng.uniform(-15, 15, m)), np.round(cy + rng.uniform(-15, 15, m))], 1)
                pix += rng.choice([0.0, 0.5], (m, 2))
            elif kind == 2:                                      # bow-tie
                a, b = rng.uniform(2, 20, 2)
                pix = np.array([[cx - a, cy - b], [cx + a, cy + b], [cx + a, cy - b], [cx - a, cy + b]])
            elif kind == 3:                                      # outside the raster, or across its border
                off = rng.choice([-1, 1]) * rng.uniform(0.5, 1.5) * (W if rng.random() < 0.5 else 0)
                ang = np.sort(rng.uniform(0, 2 * np.pi, max(m, 3)))
                rad = rng.uniform(5, 40, len(ang))
                pix = np.stack([off + cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1)
            else:                                                # star-shaped
                ang = np.sort(rng.uniform(0, 2 * np.pi, m))
                rad = rng.uniform(0.5, max(1.0, 0.4 * max(H, W)), m)
                pix = np.stack([cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1)
            ring = to_map(pix, gt)
            if rng.random() < 0.5 and len(ring) >= 3:
                ring = np.concatenate([ring, ring[:1]])
            rings.append(ring)
        polys.append(rings)
    return polys


def test_hand_made_holes_overlaps_and_brute_force(cuda):
    sq = lambda a, b: np.array([[a, a], [b, a], [b, b], [a, b]], float)     # noqa: E731
    gt = (0.0, 1.0, 0.0, 12.0, 0.0, -1.0)
    lab = assert_matches([[sq(1, 11), sq(4, 8)], [sq(5, 7)], []], gt, 12, 12)
    want = np.full((12, 12), -1, np.int32)
    want[1:11, 1:11] = 0
    want[4:8, 4:8] = -1
    want[5:7, 5:7] = 1
    assert np.array_equal(lab, want)
    rng = np.random.default_rng(1)
    H, W = 50, 70
    polys = []
    for _ in range(25):
        cx, cy = rng.uniform(0, W), rng.uniform(0, H)
        ang = np.sort(rng.uniform(0, 2 * np.pi, int(rng.integers(3, 10))))
        rad = rng.uniform(1, 12, len(ang))
        polys.append([np.stack([cx + rad * np.cos(ang), cy + rad * np.sin(ang)], 1)])
    assert_matches(polys, IDENTITY, H, W)


@pytest.mark.parametrize("transform", sorted(TRANSFORMS))
@pytest.mark.parametrize("seed", range(8))
def test_random_scenes(cuda, seed, transform):
    rng = np.random.default_rng(seed)
    gt = TRANSFORMS[transform]
    H, W = int(rng.integers(20, 160)), int(rng.integers(20, 160))
    polys = random_scene(rng, H, W, gt, int(rng.integers(5, 60)))
    kw = {}
    if seed % 2:
        kw["ids"] = rng.integers(-(1 << 31), 1 << 31, len(polys))
    if seed % 4 >= 2:
        kw["nodata"] = -7
    got = assert_matches(polys, gt, H, W, **kw)
    assert np.array_equal(gpu(shp.PolygonRings(*flat(polys)), gt, H, W, **kw), got)     # the flat form on the host


def flat(polys):
    rings = [np.asarray(r, np.float64).reshape(-1, 2) for rs in polys for r in rs]
    off = np.concatenate([[0], np.cumsum([len(r) for r in rings])]).astype(np.int64)
    rec = np.repeat(np.arange(len(polys)), [len(rs) for rs in polys]).astype(np.int32)
    xy = np.concatenate(rings) if rings else np.zeros((0, 2))
    return xy, off, rec, len(polys)


def test_flat_input_on_the_device_is_used_as_is(cuda):
    import torch
    rng = np.random.default_rng(11)
    polys = random_scene(rng, 90, 70, IDENTITY, 40)
    xy, off, rec, n = flat(polys)
    rings = shp.PolygonRings(torch.from_numpy(xy).to(cuda), torch.from_numpy(off).to(cuda), torch.from_numpy(rec).to(cuda), n)
    want = shp.rasterize_polygons(polys, IDENTITY, 90, 70, nodata=3)
    assert np.array_equal(gpu(rings, IDENTITY, 90, 70, nodata=3), want)
    assert np.array_equal(gpu(shp.PolygonRings(xy, off, rec, n), IDENTITY, 90, 70, nodata=3), want)


def test_more_crossings_than_a_sort_bucket(cuda):
    """One record with more than 4096 crossings (the bucket sort's limit per bucket): a tall rectangle and a comb."""
    H, W = 3000, 64
    rect = np.array([[2.3, -5.0], [40.7, -5.0], [40.7, H + 5.0], [2.3, H + 5.0]])
    ys = np.arange(0, H, 3, dtype=float) + 0.25
    teeth = np.concatenate([np.stack([np.full_like(ys, 5.0), ys], 1), np.stack([np.full_like(ys, 60.0), ys + 1.5], 1)], 1)
    comb = np.concatenate([teeth.reshape(-1, 2), [[0.0, H + 1.0], [0.0, -1.0]]])
    polys = [[rect], [comb], [rect[::-1] + [10, 0], comb]]
    assert crossings(polys, IDENTITY, H) > 3 * 4096
    assert_matches(polys, IDENTITY, H, W)


def test_thousands_of_tiny_polygons(cuda):
    rng = np.random.default_rng(3)
    H, W = 300, 400
    n = 6000
    c = np.stack([rng.uniform(0, W, n), rng.uniform(0, H, n)], 1)
    polys = []
    for i in range(n):
        s = rng.uniform(0.3, 2.0)
        if i % 3 == 0:
            pix = c[i] + np.array([[0, 0], [s, 0], [0, s]])
        elif i % 3 == 1:
            pix = np.floor(c[i]) + np.array([[0, 0], [s, 0], [s, s], [0, s]])   # on pixel corners
        else:
            pix = c[i] + s * np.array([[0, -1], [1, 0], [0, 1], [-1, 0]])
        polys.append([pix])
    assert_matches(polys, IDENTITY, H, W)
    assert_matches(polys, IDENTITY, H, W, ids=np.arange(n) * 7 - 5, nodata=-2)


@pytest.mark.parametrize("H,W", [(1, 37), (41, 1), (0, 9), (9, 0), (1, 1)])
def test_odd_sizes(cuda, H, W):
    rng = np.random.default_rng(H * 50 + W)
    polys = random_scene(rng, max(H, 1), max(W, 1), IDENTITY, 30)
    assert_matches(polys, IDENTITY, H, W)
    assert_matches(polys, IDENTITY, H, W, nodata=5)


def test_no_rings(cuda):
    assert_matches([[], []], IDENTITY, 5, 6)
    assert_matches([], IDENTITY, 5, 6, nodata=9)
    assert_matches([[np.array([[0.0, 0.0], [3.0, 3.0]])]], IDENTITY, 5, 6, ids=[4])


def raw(cuda, polys, gt, H, W, ld, cap, out=None, ids=None, nodata=-1):
    """dm_rasterize called directly -> (return code, counts, labels [H, ld])."""
    import torch
    from deepmerge_b200 import _lib
    L = _lib.lib()
    xy, off, rec, n = (torch.from_numpy(a).to(cuda) if isinstance(a, np.ndarray) else a for a in flat(polys))
    counts = torch.full((4,), -9, dtype=torch.int64, device=cuda)
    ws_bytes = L.dm_rasterize_workspace_bytes(xy.shape[0], n, cap)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=cuda)
    if out is None:
        out = torch.full((H, ld), 12345, dtype=torch.int32, device=cuda)
    ids_t = None if ids is None else torch.as_tensor(ids, dtype=torch.int32).to(cuda)
    rc = L.dm_rasterize(xy.data_ptr(), xy.shape[0], off.data_ptr(), rec.data_ptr(), rec.shape[0], n, gt[0], gt[1], gt[3],
                        gt[5], None if ids_t is None else ids_t.data_ptr(), nodata, H, W, ld, cap, out.data_ptr(),
                        counts.data_ptr(), ws.data_ptr(), ws_bytes, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return rc, counts.tolist(), out.cpu().numpy()


def test_strided_output_leaves_other_columns(cuda):
    rng = np.random.default_rng(21)
    H, W, ld = 70, 90, 131
    polys = random_scene(rng, H, W, IDENTITY, 40)
    n_cross = crossings(polys, IDENTITY, H)
    for kw in ({}, dict(ids=np.arange(40) + 100, nodata=-3)):
        rc, c, out = raw(cuda, polys, IDENTITY, H, W, ld, n_cross, **kw)
        assert rc == 0 and c[3] == 0 and c[2] == n_cross
        assert np.array_equal(out[:, :W], shp.rasterize_polygons(polys, IDENTITY, H, W, **kw))
        assert (out[:, W:] == 12345).all()


def test_capacity_retry_and_status(cuda):
    rng = np.random.default_rng(8)
    H, W = 120, 100
    polys = random_scene(rng, H, W, IDENTITY, 50)
    n_cross = crossings(polys, IDENTITY, H)
    assert n_cross > 64
    want = shp.rasterize_polygons(polys, IDENTITY, H, W)
    assert np.array_equal(gpu(polys, IDENTITY, H, W, capacity=64), want)
    assert np.array_equal(gpu(polys, IDENTITY, H, W, capacity=0), want)
    assert np.array_equal(gpu(polys, IDENTITY, H, W, capacity=n_cross), want)
    rc, c, _ = raw(cuda, polys, IDENTITY, H, W, W, 64)
    assert rc == 0 and c[3] == 2 and c[2] == n_cross
    rc, c, _ = raw(cuda, polys, IDENTITY, H, W, W, n_cross)
    assert rc == 0 and c[3] == 0 and c[2] == n_cross
    painted = (want >= 0).sum()
    assert c[0] > 0 and c[1] >= painted


@pytest.mark.parametrize("bad", [np.nan, np.inf, -np.inf])
@pytest.mark.parametrize("axis", [0, 1])
def test_non_finite_coordinates_raise(cuda, bad, axis):
    ring = np.array([[1.0, 1.0], [8.0, 1.5], [7.0, 9.0], [2.0, 6.0]])
    ring[2, axis] = bad
    with pytest.raises(ValueError, match="finite"):
        gpu([[ring]], IDENTITY, 10, 10)
    # a ring of fewer than 3 vertices is skipped, whatever it holds
    assert_matches([[ring[1:3]], [ring[:2] * 0 + 1]], IDENTITY, 10, 10)


def test_bad_rings_raise(cuda):
    import torch
    xy = torch.zeros((4, 2), dtype=torch.float64, device=cuda)
    with pytest.raises(ValueError, match="out of range"):
        gpu(shp.PolygonRings(xy, torch.tensor([0, 4]), torch.tensor([3], dtype=torch.int32), 2), IDENTITY, 4, 4)
    with pytest.raises(ValueError, match="out of range"):
        gpu(shp.PolygonRings(xy, torch.tensor([0, 9]), torch.tensor([0], dtype=torch.int32), 1), IDENTITY, 4, 4)
    with pytest.raises(ValueError, match="ids"):
        gpu([[xy.cpu().numpy()]], IDENTITY, 4, 4, ids=[1 << 31])
    with pytest.raises(ValueError, match="ids"):
        gpu([[xy.cpu().numpy()], []], IDENTITY, 4, 4, ids=[1])


def test_two_calls_are_bit_equal(cuda):
    rng = np.random.default_rng(5)
    polys = random_scene(rng, 400, 300, IDENTITY, 300)
    a, b = gpu(polys, IDENTITY, 400, 300), gpu(polys, IDENTITY, 400, 300)
    assert np.array_equal(a, b)


def device_rings(P, n_regions):
    """The rings of Polygons as flat device input: vertices as float64 pixel corners, one record per region."""
    return shp.PolygonRings(P.vertices.double(), P.ring_offsets, P.ring_region, n_regions)


@pytest.mark.parametrize("H,W", [(1024, 1024), (333, 517)])
def test_round_trip_voronoi_unmerged_and_merged(cuda, H, W):
    import torch
    from deepmerge_b200 import merge_scene, polygonize, rasterize
    sc = o.synth_scene(H, W, 2000 * H * W // (1024 * 1024) + 8, C=4)
    L, R = sc["labels"], sc["n_regions"]
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)    # noqa: E731
    holes = L.copy()
    holes[H // 3:H // 2, W // 4:W // 3] = -1                                     # nodata inside regions
    for lab in (L, holes):
        P = polygonize(t(lab), R)
        assert np.array_equal(rasterize(device_rings(P, R), IDENTITY, H, W).cpu().numpy(), lab)
    res = merge_scene(t(L), t(sc["feats"]), 0.5, n_regions=R, image=t(sc["image"]), xs=t(sc["xs"]), ys=t(sc["ys"]))
    P = polygonize(res.labels, R)
    assert torch.equal(rasterize(device_rings(P, R), IDENTITY, H, W), res.labels)


def test_round_trip_through_files(cuda, tmp_path):
    import torch
    from deepmerge_b200 import polygonize, rasterize
    L, R = o.synth_labels(200, 260, 300, seed=6)
    L = L.copy()
    L[40:60, 100:130] = -1
    P = polygonize(torch.from_numpy(L).to(cuda), R)
    for i, gt in enumerate([(500.0, 2.0, 0.0, 9000.0, 0.0, -2.0), (-30.0, 0.5, 0.0, 10.0, 0.0, 0.25)]):
        path = str(tmp_path / ("tile%d.shp" % i))
        shp.write_polygonized(path, P, gt)
        ids = shp.DbfTable(path[:-4] + ".dbf").column_int("REGION")
        got = rasterize(shp.read_polygon_rings(path), gt, 200, 260, ids=ids).cpu().numpy()
        assert np.array_equal(got, L)
        assert np.array_equal(got, shp.rasterize_polygons(shp.read_polygons(path), gt, 200, 260, ids=ids))


def test_round_trip_configs1_full_size(cuda):
    """configs[1] (10k x 10k, ~100k regions): the unmerged and the merged map of MergeEngine.run come back from their
    own polygons exactly.  The labels are the check; there is no host oracle at this size."""
    import torch
    from deepmerge_b200 import MergeEngine, polygonize, rasterize
    from deepmerge_b200.synth import synth_scene
    H = W = 10000
    sc = synth_scene(H, W, 100000, C=4, device=cuda)
    R = sc.n_regions
    P = polygonize(sc.labels, R)
    assert torch.equal(rasterize(device_rings(P, R), IDENTITY, H, W), sc.labels)
    eng = MergeEngine(H, W, R, sc.feats.shape[1], C=4, n_points=sc.feats.shape[0], device=cuda)
    res = eng.run(sc.labels, sc.feats, 0.5, image=sc.image, xs=sc.xs, ys=sc.ys)
    P = polygonize(res.labels, R)
    assert torch.equal(rasterize(device_rings(P, R), IDENTITY, H, W), res.labels)
