"""CPU: the oracle restatement against the golden vectors produced by EXECUTING the
reference (oracle/gen_golden.py), plus cross-checks between independent restatements for
the stages the reference has no code for (parity unpinned there)."""
import os

import numpy as np
import pytest

from oracle import golden
from oracle import oracle_np as o


def g(golden_dir, name):
    return golden.load(os.path.join(golden_dir, name))


def test_euclidean_distance_matches_reference(golden_dir):
    e = g(golden_dir, "euclid.npz")
    d = np.array([o.euclidean_distance(e["X"][i:i + 1], e["Y"][i:i + 1])[0, 0] for i in range(e["X"].shape[0])])
    assert np.array_equal(d, e["d"])                     # same numpy ops -> bit exact
    assert np.array_equal(o.euclidean_distance(e["Xm"], e["Ym"]), e["Dm"])


def test_vectorised_score_within_tolerance_of_reference(golden_dir):
    e = g(golden_dir, "euclid.npz")
    K = e["X"].shape[0]
    mean = np.concatenate([e["X"], e["Y"]])
    keys = o.pack_keys(np.arange(K), np.arange(K) + K)
    tol = o.l2_abs_tolerance(mean, keys)
    f64 = o.score_l2_f64(mean, keys)
    assert np.all(np.abs(o.score_l2(mean, keys) - f64) <= tol)
    assert np.all(np.abs(e["d"] - f64) <= tol)           # the reference itself sits inside the same band


def test_pooling_is_bit_exact_with_reference_loop(golden_dir):
    p = g(golden_dir, "pool_score.npz")
    off, ids = o.membership_csr(list(p["fields"]))
    s, c, m = o.pool_points_csr(off, ids, p["store"])
    u = p["used"]
    assert np.array_equal(m[u], p["means"][u])
    keys = (p["left"].astype(np.uint64) << np.uint64(32)) | p["right"].astype(np.uint64)
    sc = o.score_l2(m, keys)
    assert np.max(np.abs(sc - p["simi"]) / np.maximum(p["simi"], 1e-6)) < 1e-5


def test_golden_archives_split_into_parts_below_the_size_limit(golden_dir, tmp_path, monkeypatch):
    for f in os.listdir(golden_dir):
        assert os.path.getsize(os.path.join(golden_dir, f)) < golden.MAX_BYTES, f
    monkeypatch.setattr(golden, "MAX_BYTES", 3000)
    arrays = {f"a{i}": np.arange(500, dtype=np.float32) + i for i in range(3)}     # ~2.1 kB each: one per part
    path = str(tmp_path / "x.npz")
    golden.save(path, **arrays)
    assert sorted(os.listdir(tmp_path)) == ["x.1.npz", "x.2.npz", "x.npz"]
    back = golden.load(path)
    assert list(back) == list(arrays) and all(np.array_equal(back[k], arrays[k]) for k in arrays)
    golden.save(path, a0=arrays["a0"])                                             # stale parts go
    assert os.listdir(tmp_path) == ["x.npz"] and list(golden.load(path)) == ["a0"]
    with pytest.raises(ValueError, match="alone exceeds"):
        golden.save(path, big=np.zeros(1000, np.float32))


@pytest.mark.parametrize("name", ["mlp784.npz", "mlp_pair.npz"])
def test_mlp_forward_matches_nets_mlp(golden_dir, name):
    m = g(golden_dir, name)
    out, h2 = o.mlp_forward(m["x"], m["fc1_weight"], m["fc1_bias"], m["fc2_weight"], m["fc2_bias"], m["fc3_weight"],
                            m["fc3_bias"])
    np.testing.assert_allclose(out, m["fc3"], rtol=1e-4, atol=1e-5)
    np.testing.assert_allclose(h2, m["fc2"], rtol=1e-4, atol=1e-5)


def test_contrastive_loss_matches_losses_loss(golden_dir):
    l = g(golden_dir, "loss.npz")
    for mg in (1.0, 2.5):
        L, ga, gb = o.contrastive_loss(l["a"], l["b"], l["flag"], mg)
        np.testing.assert_allclose(L, l[f"loss_{mg}"], rtol=1e-6)
        np.testing.assert_allclose(ga, l[f"ga_{mg}"], rtol=1e-5, atol=1e-8)
        np.testing.assert_allclose(gb, l[f"gb_{mg}"], rtol=1e-5, atol=1e-8)


def test_edge_reader_matches_polygon_connect_dataset(golden_dir):
    e = g(golden_dir, "edge_reader.npz")
    fid, left, right = o.edges_from_lines(e["left"], e["right"])
    assert np.array_equal(fid, e["out_fid"]) and np.array_equal(left, e["out_left"]) and np.array_equal(right, e["out_right"])


def test_join_and_membership_parsers():
    assert o.neighbours_from_join("3,7,5,9", 5) == [3, 7, 9]
    off, ids = o.membership_csr(["4 2 9", "", "1"])
    assert off.tolist() == [0, 3, 3, 4] and ids.tolist() == [4, 2, 9, 1]


# ---- unpinned stages: independent restatements must agree ---------------------------------


def brute_rag(L, R):
    H, W = L.shape
    edges, area, per = {}, np.zeros(R, np.int64), np.zeros(R, np.int64)
    for y in range(H):
        for x in range(W):
            l = L[y, x]
            if l < 0:
                continue
            area[l] += 1
            for dy, dx in ((0, 1), (1, 0), (0, -1), (-1, 0)):
                yy, xx = y + dy, x + dx
                q = L[yy, xx] if 0 <= yy < H and 0 <= xx < W else -2
                if q != l:
                    per[l] += 1
                    if q >= 0 and (dy, dx) in ((0, 1), (1, 0)):
                        k = (min(l, q), max(l, q))
                        edges[k] = edges.get(k, 0) + 1
                    elif q >= 0:
                        pass
    # pairs seen from the other side (left/up) are the same pairs; count each once
    return edges, area, per


@pytest.mark.parametrize("seed", range(6))
def test_build_rag_against_brute_force(seed):
    rng = np.random.default_rng(seed)
    H, W, R = rng.integers(1, 24), rng.integers(1, 24), 9
    L = rng.integers(-1 if seed % 2 else 0, R, size=(H, W)).astype(np.int32)
    if seed == 3:
        L = np.kron(L[: (H + 3) // 4, : (W + 3) // 4], np.ones((4, 4), np.int32))[:H, :W]
    keys, blen, area, per = o.build_rag(L, R)
    edges, a2, p2 = brute_rag(L, R)
    want = sorted(edges.items())
    lo, hi = o.unpack_keys(keys)
    assert [((int(a), int(b)), int(c)) for a, b, c in zip(lo, hi, blen)] == want
    assert np.array_equal(area, a2) and np.array_equal(per, p2)
    assert np.array_equal(per, o.perimeter_by_sides(L, R))
    assert np.all(np.diff(keys.astype(np.int64)) > 0)


def test_rag_row_tiles_compose():
    sc = o.synth_scene(200, 160, 120, C=3)
    L, R = sc["labels"], sc["n_regions"]
    keys, blen, area, per = o.build_rag(L, R)
    cuts = [0, 57, 58, 131, 200]
    ks, bs = [], []
    a = np.zeros(R, np.int64)
    p = np.zeros(R, np.int64)
    for i in range(len(cuts) - 1):
        y0, y1 = cuts[i], cuts[i + 1]
        last = y1 == 200
        k, b, ai, pi = o.build_rag(L[y0:y1 + (0 if last else 1)], R, top_border=y0 == 0, bottom_border=last,
                                   own_rows=y1 - y0)
        ks.append(k); bs.append(b.astype(np.int64)); a += ai; p += pi
    uk, inv = np.unique(np.concatenate(ks), return_inverse=True)
    ub = np.bincount(inv, weights=np.concatenate(bs)).astype(np.int64)
    assert np.array_equal(uk, keys) and np.array_equal(ub, blen) and np.array_equal(a, area) and np.array_equal(p, per)


@pytest.mark.parametrize("seed", range(4))
def test_union_find_variants_agree_with_scipy(seed):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    rng = np.random.default_rng(seed)
    n, m = 200, 150
    u, v = rng.integers(0, n, m), rng.integers(0, n, m)
    a = o.union_find_min_root(n, u, v)
    b = o.min_root_propagate(n, u, v)
    assert np.array_equal(a, b)
    _, lab = connected_components(coo_matrix((np.ones(m), (u, v)), shape=(n, n)), directed=False)
    first = np.full(lab.max() + 1, n)
    np.minimum.at(first, lab, np.arange(n))
    assert np.array_equal(a, first[lab])


def test_merge_graph_invariants_and_component_backends():
    sc = o.synth_scene(160, 192, 150, C=3)
    L, R = sc["labels"], sc["n_regions"]
    a = o.merge_scene(L, R, sc["region_of_point"], sc["feats"], tau=0.5)
    keys, blen, area, per = o.build_rag(L, R)
    off, ids = o.csr_from_region_of_point(sc["region_of_point"], R)
    s, c, _ = o.pool_points_csr(off, ids, sc["feats"])
    b = o.merge_graph(s, c, area, per, keys, blen, tau=0.5, components=o.union_find_min_root)
    assert np.array_equal(a["root"], b["root"]) and a["rounds"] == b["rounds"] and a["merges"] == b["merges"]
    # merged statistics equal a fresh RAG of the relabelled raster
    k2, b2, a2, p2 = o.build_rag(a["labels"], R)
    assert np.array_equal(k2, a["keys"]) and np.array_equal(b2, a["blen"])
    roots = np.unique(a["root"])
    assert np.array_equal(a2[roots], a["area"][roots]) and np.array_equal(p2[roots], a["perim"][roots])
    assert a["merges"] == R - roots.size
    # the synthetic scene is bimodal: what merged is exactly "same ground-truth object & connected"
    assert np.all(sc["region_obj"][a["root"]] == sc["region_obj"])
    lab2, n2 = o.compact_roots(a["root"])
    assert n2 == roots.size and lab2.max() == n2 - 1


def test_multi_round_merge_chain():
    # 1-D chain 0-1-2-3 with means 0, .9, 1.7, 4: round 1 merges {0,1} (d=.9<1) and {1,2} (.8) -> one
    # component {0,1,2} mean .8667; round 2: edge to 3 has d=3.13 -> stop.  With tau=1.0.
    D = 4
    mean = np.array([0, .9, 1.7, 4.0], np.float32)[:, None].repeat(D, 1) / np.float32(2.0)   # distance = |dm|
    cnt = np.ones(4, np.int32)
    keys = o.pack_keys([0, 1, 2], [1, 2, 3])
    blen = np.array([5, 6, 7], np.uint32)
    g = o.merge_graph(mean, cnt, np.array([10, 10, 10, 10]), np.array([20, 20, 20, 20]), keys, blen, tau=1.0)
    assert g["root"].tolist() == [0, 0, 0, 3] and g["rounds"] == 1 and g["merges"] == 2
    assert g["perim"][0] == 60 - 2 * (5 + 6) and g["area"][0] == 30 and g["blen"].tolist() == [7]
    # a case that needs two rounds: 0-1 close; merged mean then comes within tau of 2
    mean = np.array([0.0, 0.8, 1.45], np.float32)[:, None].repeat(D, 1) / np.float32(2.0)
    cnt = np.array([1, 3, 1], np.int32)
    g = o.merge_graph(mean * cnt[:, None], cnt, np.ones(3, np.int64), np.full(3, 4), o.pack_keys([0, 1, 0], [1, 2, 2]),
                      np.array([1, 1, 1], np.uint32), tau=0.7)
    # round 1: d(0,1)=.8 no; d(1,2)=.65 yes; d(0,2)=1.45 no -> {1,2} mean (2.4+1.45)/4=.9625; round 2: d(0,{1,2})=.9625 no
    assert g["root"].tolist() == [0, 1, 1] and g["rounds"] == 1


def test_synth_scene_is_bimodal():
    sc = o.synth_scene(256, 256, 200, C=4)
    R = sc["n_regions"]
    keys, *_ = o.build_rag(sc["labels"], R)
    off, ids = o.csr_from_region_of_point(sc["region_of_point"], R)
    _, cnt, mean = o.pool_points_csr(off, ids, sc["feats"])
    s = o.score_l2(mean, keys)
    assert not np.any((s > 0.35) & (s < 5.0))
    lo, hi = o.unpack_keys(keys)
    same = sc["region_obj"][lo] == sc["region_obj"][hi]
    scored = (cnt[lo] > 0) & (cnt[hi] > 0)       # edge cells whose seed lies outside the image have no points
    assert scored.mean() > 0.9
    assert np.all(s[same & scored] < 0.35) and np.all(s[~same & scored] > 5.0)


def test_patch_resize_matches_the_executed_reference(golden_dir):
    """oracle.resize_area restates cv2's INTER_AREA (the arithmetic behind ExtractFeatureDataset.resize_data,
    MyUtils2.py:362-376); the golden outputs were produced by executing the reference's resize_data.  Bit exact."""
    from oracle.resize_area import resize_data
    g_ = g(golden_dir, "resize.npz")
    for i, (s, t) in enumerate(g_["cases"]):
        got = resize_data(g_[f"in{i}"], int(t))
        want = g_[f"out{i}"]
        assert got.dtype == np.float32 and got.shape == want.shape, (s, t)
        assert np.array_equal(got, want), (s, t, int((got != want).sum()))


def test_patch_resize_against_opencv_when_installed():
    """Wider sweep against cv2 itself (the reference's unpinned dependency; 4.13 in the build container)."""
    cv2 = pytest.importorskip("cv2")
    from oracle.resize_area import resize_area_u8
    rng = np.random.default_rng(9)
    for t in (32, 64, 128, 1):
        for s in sorted(set(rng.integers(2, 3 * max(t, 40), 14).tolist() + [t, 2 * t, 3 * t, 4 * t, 5 * t])):
            a = rng.integers(0, 256, (s, s), dtype=np.uint8)
            want = cv2.resize(a, (t, t), interpolation=cv2.INTER_AREA).reshape(t, t)
            assert np.array_equal(resize_area_u8(a, t), want), (s, t)


def test_reference_style_edge_loop_equals_the_executed_reference(golden_dir):
    """The per-edge loop bench.py times as the CPU arm of configs[0] reproduces the executed reference's `simi` values."""
    g = np.load(os.path.join(golden_dir, "pool_score.npz"))
    simi = o.edge_loop_reference_style(g["store"], list(g["fields"]), g["left"], g["right"])
    assert np.array_equal(simi, g["simi"])
