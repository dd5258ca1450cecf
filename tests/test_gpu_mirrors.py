"""GPU: the reference-named callables against golden vectors produced by executing the reference."""
import os

import numpy as np
import pytest

from oracle import golden
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


def test_euclidean_distance_drop_in(cuda, golden_dir):
    from deepmerge_b200.ExtractFeatures import Euclidean_distance, MC_Lyu_2020
    e = np.load(os.path.join(golden_dir, "euclid.npz"))
    D = Euclidean_distance(e["Xm"], e["Ym"])
    assert D.dtype == np.float32 and D.shape == e["Dm"].shape
    np.testing.assert_allclose(D, e["Dm"], rtol=1e-3)                       # north-star tolerance for fp32 scores
    assert np.array_equal(MC_Lyu_2020(e["Xm"], e["Ym"]), D)
    K = e["X"].shape[0]
    d = np.array([Euclidean_distance(e["X"][i:i + 1], e["Y"][i:i + 1])[0, 0] for i in range(0, K, 7)])
    mean = np.concatenate([e["X"], e["Y"]])
    keys = o.pack_keys(np.arange(0, K, 7), np.arange(0, K, 7) + K)
    assert np.all(np.abs(d - o.score_l2_f64(mean, keys)) <= o.l2_abs_tolerance(mean, keys))
    with pytest.raises(ValueError):
        Euclidean_distance(np.zeros((2, 3)), np.zeros((2, 4)))


def test_pool_and_score_matches_reference_loop(cuda, golden_dir):
    from deepmerge_b200.ExtractFeatures import pool_and_score
    p = np.load(os.path.join(golden_dir, "pool_score.npz"))
    means, simi = pool_and_score(p["store"], list(p["fields"]), p["left"], p["right"])
    u = p["used"]
    assert np.array_equal(means[u], p["means"][u])                          # np.mean(axis=0), bit exact
    assert simi.dtype == np.float64
    np.testing.assert_allclose(simi, p["simi"], rtol=1e-3)


def test_loss_forward_backward_matches_reference(cuda, golden_dir):
    import torch
    from deepmerge_b200.Losses import Loss
    l = np.load(os.path.join(golden_dir, "loss.npz"))
    for mg in (1.0, 2.5):
        a = torch.from_numpy(l["a"]).to(cuda).requires_grad_(True)
        b = torch.from_numpy(l["b"]).to(cuda).requires_grad_(True)
        loss = Loss(mg, 0.1, 0)(a, b, torch.from_numpy(l["flag"]).to(cuda))
        (3.0 * loss).backward()                                             # upstream gradient is honoured
        np.testing.assert_allclose(loss.item(), l[f"loss_{mg}"], rtol=1e-5)
        np.testing.assert_allclose(a.grad.cpu().numpy(), 3.0 * l[f"ga_{mg}"], rtol=1e-5, atol=1e-8)
        np.testing.assert_allclose(b.grad.cpu().numpy(), 3.0 * l[f"gb_{mg}"], rtol=1e-5, atol=1e-8)
    with pytest.raises(ValueError):
        Loss(1.0, 0.1, 0)(torch.zeros(2, 3), torch.zeros(2, 3), torch.zeros(2))


def test_pair_training_step_gather_plus_loss(cuda):
    """R10 + R11 together: sampled point pairs -> gathered embedding rows -> loss + grads."""
    import torch
    from deepmerge_b200._lib import lib
    from deepmerge_b200.Losses import Loss
    rng = np.random.default_rng(3)
    table = rng.standard_normal((500, 100)).astype(np.float32)
    left, right = rng.integers(0, 500, 960), rng.integers(0, 500, 960)
    flag = rng.integers(0, 2, 960)
    L = lib()
    t = torch.from_numpy(table).to(cuda)
    ga = torch.empty((960, 100), device=cuda)
    gb = torch.empty((960, 100), device=cuda)
    L.check(L.dm_gather_rows(t.data_ptr(), 100, torch.from_numpy(left).to(cuda).data_ptr(), 960, ga.data_ptr(), None), "g")
    L.check(L.dm_gather_rows(t.data_ptr(), 100, torch.from_numpy(right).to(cuda).data_ptr(), 960, gb.data_ptr(), None), "g")
    assert np.array_equal(ga.cpu().numpy(), table[left]) and np.array_equal(gb.cpu().numpy(), table[right])
    loss = Loss(1.0, 0.1, 0)(ga.requires_grad_(True), gb, torch.from_numpy(flag).to(cuda))
    want, wga, _ = o.contrastive_loss(table[left], table[right], flag, 1.0)
    np.testing.assert_allclose(loss.item(), want, rtol=1e-5)
    loss.backward()
    np.testing.assert_allclose(ga.grad.cpu().numpy(), wga, rtol=1e-4, atol=1e-8)


def test_cut_windows_matches_reference_cutter(cuda, golden_dir):
    """N1 first piece: the batched GPU window cut reproduces ExtractFeatureDataset.cut_image (executed reference,
    golden geometry.npz) bit for bit, including windows that hang over every border and a 1 x 1 window."""
    import torch
    from deepmerge_b200 import MyUtils2 as m
    g = np.load(os.path.join(golden_dir, "geometry.npz"))
    img = torch.from_numpy(g["arr"]).to(cuda)
    for i, (x, y, w) in enumerate(g["mids"]):
        got = m.cut_windows(img, [int(x)], [int(y)], int(w))[0].cpu().numpy()
        assert np.array_equal(got, g[f"cut{i}"]), i
    # a batch of same-sized windows against the host mirror of the cutter
    rng = np.random.default_rng(0)
    xs, ys = rng.integers(-5, 56, size=64), rng.integers(-5, 46, size=64)
    got = m.cut_windows(img, xs, ys, 9).cpu().numpy()
    for k in range(64):
        win = m.calculate_left_top_point_and_size(int(xs[k]), int(ys[k]), 9)
        assert np.array_equal(got[k], m.cut_image(g["arr"], win))


def test_test_for_shp_on_real_shapefiles(cuda, golden_dir, tmp_path, capsys):
    """The reference's test_for_shp (ExtractFeatures.py:150-225) end to end on files on disk: attribute tables read
    without GDAL, pooling + scoring on the GPU, `simi` written back as an OFTReal attribute of every kept line."""
    from deepmerge_b200 import shapefile
    from deepmerge_b200.ExtractFeatures import FeatureIO, test_for_shp
    p = np.load(os.path.join(golden_dir, "pool_score.npz"))
    d = tmp_path / "tile"
    d.mkdir()
    left, right = p["left"].copy(), p["right"].copy()
    right[7] = -1
    shapefile.write_dbf(str(tmp_path / "tile.dbf"), [("PointID", "C", 60, 0)], {"PointID": list(p["fields"])})
    shapefile.write_dbf(str(d / "lines.dbf"), [("LEFT_FID", "N", 9, 0), ("RIGHT_FID", "N", 9, 0)],
                        {"LEFT_FID": left, "RIGHT_FID": right})
    shapefile.write_dbf(str(d / "PointsGCS.dbf"), [("inner", "N", 9, 0)], {"inner": np.arange(len(p["store"]))})
    np.save(tmp_path / "feats.npy", p["store"])
    io = FeatureIO()
    io.ReadFeatures(str(tmp_path / "feats.npy"))
    assert test_for_shp(io, None, str(tmp_path / "tile.shp"), str(d / "lines.shp"), str(d / "PointsGCS.shp")) == 0
    col = shapefile.DbfTable(str(d / "lines.dbf")).column_float("simi")
    keep = np.arange(len(left)) != 7
    assert np.isnan(col[7])
    np.testing.assert_allclose(col[keep], p["simi"][keep], rtol=1e-3)


def test_pair_dataset_items_equal_the_executed_reference(cuda, golden_dir, tmp_path):
    """ds[i] -> (left_meta, right_meta, flag), meta = (designed [1,19], scales [1,4], [4 patches]): every item of the
    executed reference class (MyUtils1.py:41-80, patches through cv2 INTER_AREA) bit for bit, and batch() == items."""
    import random
    import torch
    from deepmerge_b200 import MyUtils1
    from test_mirrors_cpu import _pair_dataset_fixture
    g = golden.load(os.path.join(golden_dir, "pair_dataset.npz"))
    pos, neg, open_vector, open_image = _pair_dataset_fixture(g, tmp_path)
    random.seed(int(g["seed"]))
    ds = MyUtils1.MergingSegmensPairDataset("IF", "PF", "QF", pos, neg, open_vector=open_vector, open_image=open_image,
                                            device=cuda)
    n = int(g["n"])
    for i in range(n):
        left, right, flag = ds[i]
        assert flag == int(g[f"flag{i}"])
        for side, meta in (("l", left), ("r", right)):
            assert isinstance(meta[0], torch.Tensor) and tuple(meta[0].shape) == (1, 19) and tuple(meta[1].shape) == (1, 4)
            assert np.array_equal(meta[0].numpy(), g[f"{side}{i}_designed"])
            assert np.array_equal(meta[1].numpy(), g[f"{side}{i}_scales"])
            for k in range(4):
                assert meta[2][k].dtype == np.float32 and np.array_equal(meta[2][k], g[f"{side}{i}_patch{k}"]), (i, side, k)
    b = ds.batch(range(n))
    assert b["flag"].tolist() == [int(g[f"flag{i}"]) for i in range(n)]
    for side, key in (("l", "left"), ("r", "right")):
        designed, scales, patches = b[key]
        assert np.array_equal(designed.cpu().numpy(), np.concatenate([g[f"{side}{i}_designed"] for i in range(n)]))
        for k in range(4):
            assert np.array_equal(patches[k].cpu().numpy(), np.stack([g[f"{side}{i}_patch{k}"] for i in range(n)]))


def test_join_adjacency_drives_the_merge_loop(cuda):
    """R2: the polygon `join` fields (MyUtils.py:110-114, neighbour ids including self) parsed by edge_keys_from_join give
    the graph build_rag extracts from the raster; merge_graph on it equals the oracle."""
    import torch
    from deepmerge_b200 import MyUtils, merge_graph
    from oracle import oracle_np as o
    sc = o.synth_scene(160, 256, 260, C=4)
    R = sc["n_regions"]
    keys, blen, area, per = o.build_rag(sc["labels"], R)
    lo, hi = o.unpack_keys(keys)
    nb = [[r] for r in range(R)]
    for a, b in zip(lo.tolist(), hi.tolist()):
        nb[a].append(b)
        nb[b].append(a)
    join = [",".join(str(v) for v in sorted(l)) for l in nb]                  # the attribute as the reference reads it
    assert MyUtils.neighbours_from_join(join[5], 5) == sorted(v for v in nb[5] if v != 5)
    jk = MyUtils.edge_keys_from_join(join)
    assert np.array_equal(jk.view(np.uint64), keys)
    off, ids = o.csr_from_region_of_point(sc["region_of_point"], R)
    ps, cnt, _ = o.pool_points_csr(off, ids, sc["feats"])
    want = o.merge_graph(ps, cnt, area, per, keys, blen, tau=0.5)
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    got = merge_graph(T(ps), T(cnt), T(area), T(per), T(jk), T(blen.view(np.int32)), 0.5)
    assert np.array_equal(got.root.cpu().numpy(), want["root"]) and got.rounds == want["rounds"] and got.merges == want["merges"]
    assert np.array_equal(got.edge_keys.cpu().numpy().view(np.uint64), want["keys"])


@pytest.mark.parametrize("shape", [(96, 128, 40), (257, 301, 150), (1030, 777, 2000)])
def test_designed_attributes_on_the_device(cuda, shape):
    """N2: RAG.attributes() from a device pass -- bounding boxes bit for bit against the oracle, the attributes against
    oracle_np.shape_attributes / the pixels themselves (float32 of the same float64 expression)."""
    import torch
    from deepmerge_b200 import raster as rs
    H, W, n = shape
    sc = o.synth_scene(H, W, n, C=4, seed=H)
    R = sc["n_regions"] + 3                                   # three ids without pixels
    lab = sc["labels"].copy()
    lab[5:9, 7:19] = -1                                       # a nodata hole
    d_lab = torch.from_numpy(lab).cuda()
    rag = rs.build_rag(d_lab, R, torch.from_numpy(sc["image"]).cuda(), bbox=True)
    box = o.region_bbox(lab, R)
    assert np.array_equal(rag.bbox.cpu().numpy(), box)
    assert np.array_equal(rs.region_bbox(d_lab, R).cpu().numpy(), box)
    area, perim = o.build_rag(lab, R)[2:4]
    want = o.shape_attributes(area, perim, box)
    a = {k: v.cpu().numpy() for k, v in rag.attributes().items()}
    for k, v in want.items():
        np.testing.assert_allclose(a[k], v, rtol=1e-6, equal_nan=True, err_msg=k)
    assert np.isnan(a["len"][-3:]).all() and np.array_equal(a["area"], area.astype(np.float32))
    r = int(np.argmax(area))
    ys, xs = np.nonzero(lab == r)
    assert a["len"][r] == max(np.ptp(xs), np.ptp(ys)) + 1 and a["width"][r] == min(np.ptp(xs), np.ptp(ys)) + 1
    with pytest.raises(ValueError):
        rs.region_bbox(d_lab, R - 10)
