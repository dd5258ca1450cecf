"""CPU: host-side mirrors of the reference's Python interface against golden vectors produced by
executing the reference (edge-list reader, pair sampler)."""
import os
import random

import numpy as np
import pytest

from deepmerge_b200 import MyUtils1, MyUtils2
from oracle import golden
from oracle.ref_shim import FakeFeature, FakeLayer, FakeRaster


def test_edge_reader_matches_reference(golden_dir, capsys):
    e = np.load(os.path.join(golden_dir, "edge_reader.npz"))
    lines = FakeLayer([FakeFeature(i, {"LEFT_FID": int(l), "RIGHT_FID": int(r)}) for i, (l, r) in
                       enumerate(zip(e["left"], e["right"]))])
    ds = MyUtils2.PolygonConnectPointDataset("X:\\img\\tileA.tif", "X:\\tiles\\tileA.shp", "X:\\tiles\\tileA\\lines.shp",
                                             "X:\\tiles\\tileA\\PointsGCS.shp", line_layer=lines, polygon_layer=FakeLayer([]),
                                             point_layer=FakeLayer([]), img_dataset=FakeRaster(np.zeros((3, 8, 8), np.uint8)))
    assert len(ds) == len(e["out_fid"])
    rows = [ds[i] for i in range(len(ds))]
    assert [r[0] for r in rows] == e["out_fid"].tolist() and [r[1] for r in rows] == e["out_name"].tolist()
    assert [r[2] for r in rows] == e["out_left"].tolist() and [r[3] for r in rows] == e["out_right"].tolist()
    keys = ds.edge_keys()
    assert np.array_equal(keys >> 32, np.minimum(e["out_left"], e["out_right"]))
    assert ds.band_num == 3 and ds.line_layer is lines


def test_edge_reader_without_gdal_raises_like_the_reference():
    import pytest
    with pytest.raises(ValueError, match="Can not open"):
        MyUtils2.PolygonConnectPointDataset("a.tif", "a.shp", "lines.shp", "pts.shp")


def test_pair_sampler_reproduces_reference_under_the_same_seed(golden_dir, tmp_path):
    g = np.load(os.path.join(golden_dir, "pair_sampler.npz"))
    fields = list(g["fields"])
    p = tmp_path / "tileP.txt"
    p.write_text("".join(f"{j},{a},{b},0,0\n" for j, (a, b) in enumerate(g["pos_pairs"])))
    pairs = MyUtils1.read_pair_list(str(p))
    assert [[int(a), int(b)] for a, b in pairs] == g["pos_pairs"].tolist()
    random.seed(int(g["seed"]))
    data = MyUtils1.sample_pairs(fields, pairs, 1, "tileP") + MyUtils1.sample_pairs(fields, g["neg_pairs"].tolist(), 0, "tileN")
    left, right, flag = MyUtils1.pairs_to_arrays(data)
    assert np.array_equal(left, g["out_left"]) and np.array_equal(right, g["out_right"]) and np.array_equal(flag, g["out_flag"])
    assert [d[0] for d in data] == g["out_tile"].tolist()
    assert g["counts"].tolist() == [len(g["pos_pairs"]), len(g["pos_pairs"]), len(g["neg_pairs"]), len(g["neg_pairs"])]


def test_geometry_helpers_match_reference_golden(golden_dir):
    """R12: pixel mapping (+1), window placement, scale factors and the zero-padded cutter against values
    produced by executing MyUtils2.ExtractFeatureDataset (oracle/gen_golden.py:golden_geometry)."""
    from deepmerge_b200 import MyUtils2 as m
    g = np.load(os.path.join(golden_dir, "geometry.npz"))
    px, ln = m.geo_to_pixel(tuple(g["gt"]), g["geo"][:, 0], g["geo"][:, 1])
    assert np.array_equal(np.stack([px, ln], 1), g["px"])
    for (x, y, w), want in zip(g["mids"], g["wins"]):
        assert m.calculate_left_top_point_and_size(int(x), int(y), int(w)) == tuple(int(v) for v in want)
    left, top, w, h = m.calculate_left_top_point_and_size(g["mids"][:, 0], g["mids"][:, 1], g["mids"][:, 2])
    assert np.array_equal(np.stack([left, top, w, h], 1), g["wins"])
    assert tuple(g["cfg_scales"]) == m.SCALES
    for (a, b), s, f in zip(g["io"], g["scales"], g["factors"]):
        sc, fa = m.get_scales(int(a), int(b))
        assert sc == [int(v) for v in s] and np.allclose(fa, f, rtol=0, atol=0)
    for i, win in enumerate(g["wins"]):
        assert np.array_equal(m.cut_image(g["arr"], win), g[f"cut{i}"])


def test_join_adjacency_form():
    """R2: `join` lists include the polygon itself (MyUtils.py:110-114); keys come out canonical."""
    from deepmerge_b200 import MyUtils as m
    from oracle import oracle_np as o
    joins = ["0,1,2", "0,1", "2,0,3", "3,2"]
    assert m.neighbours_from_join(joins[2], 2) == o.neighbours_from_join(joins[2], 2) == [0, 3]
    keys = m.edge_keys_from_join(joins)
    assert np.array_equal(keys.view(np.uint64), o.pack_keys(np.array([0, 0, 2]), np.array([1, 2, 3])))
    with pytest.raises(ValueError):
        m.neighbours_from_join("1,2", 5)            # self missing: list.remove raises like the reference
    off, ids = m.membership_from_points(["4,9", "", "7"])
    assert off.tolist() == [0, 2, 2, 3] and ids.tolist() == [4, 9, 7]


def test_checkpoint_dictionary_round_trip(tmp_path):
    """Train_SMT.py:318-340 / :164-198: keys, file-name pattern, resume of network + optimizer state."""
    import time
    import torch
    from deepmerge_b200 import checkpoint
    from deepmerge_b200.Nets import MLP
    torch.manual_seed(0)
    net = MLP(dims=(200, 250, 2))
    net.name, net.depth, net.input_image_scales = "pairMLP", 3, [32, 64, 128, 1]
    opt = torch.optim.SGD(net.parameters(), lr=0.1, momentum=0.9)
    net.fc1.weight.grad = torch.ones_like(net.fc1.weight)
    opt.step()
    t = time.struct_time((2024, 3, 9, 14, 5, 0, 0, 0, 0))
    assert checkpoint.model_name(99, t) == "model-2024-3-9_14-5_100epochs.pth"
    p = checkpoint.save(str(tmp_path / checkpoint.model_name(4, t)), net, opt, 4, 123.456)
    raw = torch.load(p, weights_only=False)
    assert tuple(raw.keys()) == checkpoint.KEYS and raw["time"] == 123.46 and raw["epoch"] == 4
    assert raw["name"] == "pairMLP" and raw["depth"] == 3 and raw["scales"] == [32, 64, 128, 1]
    net2 = MLP(dims=(200, 250, 2))
    opt2 = torch.optim.SGD(net2.parameters(), lr=0.1, momentum=0.9)
    ck = checkpoint.load(p, net2, opt2)
    assert ck["epoch"] == 4 and all(torch.equal(a, b) for a, b in zip(net.state_dict().values(), net2.state_dict().values()))
    assert torch.equal(opt2.state_dict()["state"][0]["momentum_buffer"], opt.state_dict()["state"][0]["momentum_buffer"])
    # a bare state_dict (the reference's `weights` argument) loads too
    torch.save(net.state_dict(), str(tmp_path / "weights.pth"))
    net3 = MLP(dims=(200, 250, 2))
    assert checkpoint.load(str(tmp_path / "weights.pth"), net3)["epoch"] == -1
    assert torch.equal(net3.fc3.bias, net.fc3.bias)


def test_area_tables_agree_with_the_oracle_restatement():
    """The product's host-side table builder (what dm_resize_area consumes) and the oracle's independent restatement
    of OpenCV's INTER_AREA rules give the same tables for every (source, target) size the loader can meet."""
    from oracle import resize_area as ora
    for t in (32, 64, 128, 1):
        for s in range(1, 3 * max(t, 40)):
            mode, ti, tf = MyUtils2.area_tables(s, t)
            if s % t == 0:
                assert mode == 0 and ti is None and tf is None
            elif s > t:
                di, si, al = ora._area_table(s, t)
                start = np.searchsorted(np.asarray(di), np.arange(t + 1))
                assert mode == 1 and np.array_equal(ti[:t + 1], start) and np.array_equal(ti[t + 1:], si)
                assert tf.dtype == np.float32 and np.array_equal(tf, np.asarray(al, np.float32))
            else:
                sx, a0, a1, xmax = ora._linear_table(s, t)
                assert mode == 2 and np.array_equal(ti, np.concatenate([sx, a0, a1, [xmax]]))


def test_rag_attributes_from_the_pooled_statistics():
    """RAG.attributes(): area / peri / mean / std / bright of every region from the integer sums of the raster pass
    (device-agnostic tensor arithmetic; the sums themselves are checked bit-exactly by the GPU parity tests)."""
    import torch
    from deepmerge_b200.raster import RAG
    from oracle import oracle_np as o
    sc = o.synth_scene(96, 128, 40, C=3)
    R = sc["n_regions"]
    s, q = o.pool_bands(sc["labels"], sc["image"], R)
    keys, blen, area, perim = o.build_rag(sc["labels"], R)[:4]
    rag = RAG(torch.from_numpy(keys.view(np.int64)), torch.from_numpy(blen.view(np.int32)), torch.from_numpy(area),
              torch.from_numpy(perim), torch.zeros(R, dtype=torch.int64), torch.from_numpy(s.view(np.int64)),
              torch.from_numpy(q.view(np.int64)))
    a = rag.attributes()
    for r in range(R):
        px = sc["image"][sc["labels"] == r].astype(np.float64)
        assert a["area"][r].item() == len(px) and a["peri"][r].item() == perim[r]
        if len(px):
            np.testing.assert_allclose(a["mean"][r].numpy(), px.mean(axis=0), rtol=1e-6)
            np.testing.assert_allclose(a["std"][r].numpy(), px.std(axis=0), rtol=1e-5, atol=1e-4)
            np.testing.assert_allclose(a["bright"][r].item(), px.mean(axis=0).mean(), rtol=1e-6)
        else:
            assert torch.isnan(a["mean"][r]).all()
    rag.bbox = torch.from_numpy(o.region_bbox(sc["labels"], R))
    a = rag.attributes()
    want = o.shape_attributes(area, perim, rag.bbox.numpy())
    for k, v in want.items():
        np.testing.assert_allclose(a[k].numpy(), v, rtol=1e-6, equal_nan=True, err_msg=k)
    for r in range(0, R, 7):
        ys, xs = np.nonzero(sc["labels"] == r)
        if len(ys):
            w, h = np.ptp(xs) + 1, np.ptp(ys) + 1
            assert a["len"][r].item() == max(w, h) and a["width"][r].item() == min(w, h)
            np.testing.assert_allclose(a["compact"][r].item(), w * h / len(ys), rtol=1e-6)


def test_point_patches_grouping_logic(monkeypatch):
    """point_patches groups the points by window size and scatters every group's patches back in point order.  The
    two GPU calls are replaced by host stand-ins here (cut_image per point, the oracle resize), so that the grouping
    itself is checked without a device; the real kernels are covered by tests/test_zz_gpu_resize.py."""
    import torch
    from oracle.resize_area import resize_data
    rng = np.random.default_rng(8)
    img = rng.integers(0, 256, (2, 90, 110), dtype=np.uint8)

    def fake_cut(image, xpix, ylin, size):
        a = image.numpy()
        return torch.from_numpy(np.stack([MyUtils2.cut_image(a, MyUtils2.calculate_left_top_point_and_size(int(x), int(y), size))
                                          for x, y in zip(xpix, ylin)]))

    def fake_resize(windows, t):
        return torch.from_numpy(np.stack([resize_data(w, t) for w in windows.numpy()]))

    monkeypatch.setattr(MyUtils2, "cut_windows", fake_cut)
    monkeypatch.setattr(MyUtils2, "resize_windows", fake_resize)
    n = 10
    inner, obj = rng.integers(6, 12, n), rng.integers(14, 20, n)          # few distinct sizes -> real groups
    scales = np.stack([inner, obj, 2 * obj - inner, 3 * obj - 2 * inner], axis=1)
    w = {"ids": np.arange(n), "scales": scales, "xpix": rng.integers(1, 111, n), "ylin": rng.integers(1, 91, n)}
    got = MyUtils2.point_patches(torch.from_numpy(img), w)
    for k, cfg in enumerate(MyUtils2.SCALES):
        assert tuple(got[k].shape) == (n, 2, cfg, cfg)
        for i in range(n):
            win = MyUtils2.calculate_left_top_point_and_size(int(w["xpix"][i]), int(w["ylin"][i]), int(scales[i, k]))
            assert np.array_equal(got[k][i].numpy(), resize_data(MyUtils2.cut_image(img, win), cfg)), (i, k)


def test_pool_and_score_rejects_ids_outside_the_store_before_touching_the_gpu():
    """ExtractFeatures.py:109-112: a row outside the feature store is an error in the reference; here the ids are
    validated on the host because the kernels gather by them without bounds tests."""
    from deepmerge_b200.ExtractFeatures import check_ids, pool_and_score
    store = np.zeros((5, 4), np.float32)
    with pytest.raises(IndexError):
        pool_and_score(store, ["0 1", "2 7"], [0], [1])                    # PointID 7 >= 5 rows
    with pytest.raises(IndexError):
        pool_and_score(store, ["0 1", "2 3"], [0], [2])                    # RIGHT_FID 2: only polygons 0 and 1 exist
    with pytest.raises(IndexError):
        check_ids(np.array([-1, 0]), 5, [0], [1], 2)
    check_ids(np.array([0, 4]), 5, [0, 1], [1, 0], 2)                      # in range: no error


def _pair_dataset_fixture(g, tmp_path):
    """Fake OGR / GDAL objects and the two pair-list folders the golden generator used (oracle/gen_golden.py)."""
    from deepmerge_b200.MyUtils2 import DESIGNED_FIELDS
    fields = list(g["fields"])
    polys = FakeLayer([FakeFeature(r, {"PointID": fields[r]}) for r in range(len(fields))])

    def point(i):
        f = dict(zip(DESIGNED_FIELDS, g["attr"][i].tolist()))
        f["inner"], f["object"] = int(g["inner"][i]), int(g["obj"][i])
        return FakeFeature(i, f, (float(g["X"][i]), float(g["Y"][i])))

    pts = FakeLayer([point(i) for i in range(len(g["X"]))])
    pos, neg = tmp_path / "pos", tmp_path / "neg"
    pos.mkdir()
    neg.mkdir()
    (pos / "tileA.txt").write_text("".join(f"{j},{a},{b},0,0\n" for j, (a, b) in enumerate(g["pos_pairs"])))
    (neg / "tileB.txt").write_text("".join(f"{j},{a},{b},0,0\n" for j, (a, b) in enumerate(g["neg_pairs"])))

    class DS:
        def __init__(self, layer):
            self.layer = layer

        def GetLayer(self, i):
            return self.layer

    def open_vector(path):
        layer = pts if path.endswith("PointsGCS.shp") else polys
        return DS(layer), layer

    def open_image(path):
        return FakeRaster(g["arr"], geotransform=tuple(g["gt"]))

    return str(pos), str(neg), open_vector, open_image


def test_pair_dataset_class_builds_the_reference_item_list(golden_dir, tmp_path):
    """MergingSegmensPairDataset(image_folder, polygon_folder, point_folder, positive_folder, negative_folder): same
    attributes and, under the same seed, the item list of the executed reference (MyUtils1.py:20-38, :236-295)."""
    g = golden.load(os.path.join(golden_dir, "pair_dataset.npz"))
    pos, neg, open_vector, open_image = _pair_dataset_fixture(g, tmp_path)
    random.seed(int(g["seed"]))
    ds = MyUtils1.MergingSegmensPairDataset("IF", "PF", "QF", pos, neg, open_vector=open_vector, open_image=open_image)
    assert len(ds) == int(g["n"])
    assert [ds.positive_number, ds.positive_pair_number, ds.negative_number, ds.negative_pair_number] == g["counts"].tolist()
    assert [[d[0], str(d[1]), str(d[2]), str(d[3])] for d in ds.data] == g["data"].tolist()
    assert set(ds.layers) == {"tileA", "tileB"} and set(ds.img_dataset) == {"tileA", "tileB"} and ds.band_num == 3
    empty = MyUtils1.MergingSegmensPairDataset("IF", "PF", "QF", "", "", open_vector=open_vector, open_image=open_image)
    assert len(empty) == 0 and empty.positive_pair_number == 0
