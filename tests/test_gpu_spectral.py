"""GPU: merge by spectral and shape heterogeneity, bit for bit against the oracle (tests/spectral_oracle.py: spectral_fusion,
select_mutual, merge_spectral): the score kernel on random graphs, the mutual best selection on its edge cases, the
integer merge of the statistics, and the whole run_spectral loop on synthetic scenes up to the configs[1] size."""
import numpy as np
import pytest
import torch

from oracle import oracle_np as o

import spectral_oracle as so
from test_spectral_core_cpu import random_stats

pytestmark = pytest.mark.gpu

SENTINEL = np.float32(-12345.5)


def T(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def I64(a, dev):
    return T(np.asarray(a).view(np.int64) if np.asarray(a).dtype == np.uint64 else np.asarray(a, np.int64), dev)


def bits(x):
    x = x.cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return np.asarray(x, np.float32).view(np.uint32)


def u64(t):
    return t.cpu().numpy().view(np.uint64)


@pytest.fixture(scope="module")
def L(cuda):
    from deepmerge_b200 import _lib
    return _lib.lib()


def stream():
    return torch.cuda.current_stream().cuda_stream


def score_dev(L, g, dev, w_shape, w_cmpct, band_w=None, rescore=None, init=None):
    E = g["keys"].shape[0]
    keys, blen = I64(g["keys"], dev), T(g["blen"].view(np.int32), dev)
    area, perim = I64(g["area"], dev), I64(g["perim"], dev)
    bsum, bsq, box = I64(g["bsum"], dev), I64(g["bsq"], dev), T(g["bbox"], dev)
    n = torch.tensor([E], dtype=torch.int64, device=dev)
    out = T(np.full(E, SENTINEL, np.float32) if init is None else init, dev)
    bw = None if band_w is None else T(np.asarray(band_w, np.float32), dev)
    rs = None if rescore is None else T(rescore.astype(np.uint8), dev)
    L.check(L.dm_score_spectral(keys.data_ptr(), blen.data_ptr(), n.data_ptr(), E, area.data_ptr(), perim.data_ptr(),
                                bsum.data_ptr(), bsq.data_ptr(), g["bsum"].shape[1], box.data_ptr(),
                                None if bw is None else bw.data_ptr(), w_shape, w_cmpct,
                                None if rs is None else rs.data_ptr(), out.data_ptr(), stream()), "dm_score_spectral")
    return out.cpu().numpy()


@pytest.mark.parametrize("C", [1, 3, 4, 8])
def test_score_spectral_bit_exact_on_random_graphs(L, cuda, C):
    rng = np.random.default_rng(40 + C)
    R = 5000
    g = random_stats(rng, R, C, 60000)
    bw = (rng.random(C) * 2).astype(np.float32)
    for w_shape, w_cmpct, band_w in ((0.1, 0.5, None), (0.9, 0.0, bw), (1.0, 1.0, None), (0.0, 0.5, bw)):
        want = so.spectral_fusion(g["area"], g["perim"], g["bsum"], g["bsq"], g["bbox"], g["keys"], g["blen"], w_shape,
                                 w_cmpct, band_w)
        assert np.array_equal(bits(score_dev(L, g, cuda, w_shape, w_cmpct, band_w)), bits(want)), (w_shape, w_cmpct)
        # rescore mask: only edges with a flagged endpoint are recomputed, the others keep their value
        flag = rng.random(R) < 0.1
        lo, hi = o.unpack_keys(g["keys"])
        touched = flag[lo] | flag[hi]
        init = rng.standard_normal(len(lo)).astype(np.float32)
        got = score_dev(L, g, cuda, w_shape, w_cmpct, band_w, rescore=flag, init=init)
        assert 0 < touched.sum() < len(lo)
        assert np.array_equal(bits(got[touched]), bits(want[touched])) and np.array_equal(bits(got[~touched]), bits(init[~touched]))


def test_score_spectral_stage_entry_on_a_scene(cuda):
    from deepmerge_b200 import build_rag, score_spectral
    sc = o.synth_scene(300, 400, 700, C=3)
    rag = build_rag(T(sc["labels"], cuda), sc["n_regions"], T(sc["image"], cuda), bbox=True)
    keys, blen, area, perim = o.build_rag(sc["labels"], sc["n_regions"])
    s, q = o.pool_bands(sc["labels"], sc["image"], sc["n_regions"])
    box = o.region_bbox(sc["labels"], sc["n_regions"])
    for kw in (dict(), dict(shape=0.5, compactness=0.2, band_weights=[1.0, 0.5, 2.0])):
        want = so.spectral_fusion(area, perim, s, q, box, keys, blen, kw.get("shape", 0.1), kw.get("compactness", 0.5),
                                 kw.get("band_weights"))
        assert np.array_equal(bits(score_spectral(rag, **kw)), bits(want))


def select_dev(L, scores, keys, thr, R, dev, cap=None):
    E = len(keys)
    cap = max(E, 1) if cap is None else cap
    s = T(np.r_[np.asarray(scores, np.float32), np.zeros(cap - E, np.float32)], dev)
    k = T(np.r_[np.asarray(keys, np.uint64), np.zeros(cap - E, np.uint64)].view(np.int64), dev)
    n = torch.tensor([E], dtype=torch.int64, device=dev)
    sel = torch.full((cap,), 7, dtype=torch.uint8, device=dev)
    cnt = torch.full((1,), -1, dtype=torch.int64, device=dev)
    wsb = L.dm_merge_select_mutual_workspace_bytes(R)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    L.check(L.dm_merge_select_mutual(s.data_ptr(), float(thr), k.data_ptr(), n.data_ptr(), cap, R, sel.data_ptr(),
                                     cnt.data_ptr(), ws.data_ptr(), wsb, stream()), "dm_merge_select_mutual")
    sel = sel.cpu().numpy()
    assert (sel[E:] == 7).all()                                    # nothing written past the live edges
    return sel[:E].astype(bool), int(cnt.item())


def check_select(L, scores, keys, thr, R, dev):
    want = so.select_mutual(scores, keys, thr, R)
    got, n = select_dev(L, scores, keys, thr, R, dev)
    assert np.array_equal(got, want) and n == int(want.sum())
    return want


def test_select_mutual_edge_cases(L, cuda):
    rng = np.random.default_rng(5)
    R = 3000
    a = rng.integers(0, R - 1, 20000)
    b = a + 1 + (rng.random(20000) * (R - 1 - a)).astype(np.int64)
    keys = np.unique(o.pack_keys(a, b))
    E = len(keys)
    # ties: a handful of distinct values, so most minima are decided by the edge index
    ties = rng.integers(0, 4, E).astype(np.float32)
    want = check_select(L, ties, keys, 10.0, R, cuda)
    assert want.sum() > 10
    # NaN, negative values, both zeros, infinities
    s = rng.standard_normal(E).astype(np.float32) * 100
    s[rng.random(E) < 0.2] = np.nan
    s[rng.random(E) < 0.05] = -0.0
    s[rng.random(E) < 0.05] = 0.0
    s[rng.random(E) < 0.02] = -np.inf
    want = check_select(L, s, keys, 50.0, R, cuda)
    assert not want[np.isnan(s)].any() and want.sum() > 10
    # a threshold exactly equal to scores: those edges are not below it
    s = (5 + rng.integers(0, 3, E)).astype(np.float32)
    assert not check_select(L, s, keys, 5.0, R, cuda).any()
    assert check_select(L, s, keys, np.nextafter(np.float32(5), np.float32(6)), R, cuda).sum() > 10
    # a hub region with thousands of edges, its best edge tied with others
    hub_keys = o.pack_keys(np.zeros(5000, np.int64), np.arange(1, 5001))
    spoke = o.pack_keys(np.arange(1, 5000), np.arange(2, 5001))
    k = np.unique(np.r_[hub_keys, spoke])
    s = (rng.integers(0, 3, len(k)) + 1).astype(np.float32)
    want = check_select(L, s, k, 100.0, 5001, cuda)
    lo, hi = o.unpack_keys(k)
    assert want[lo == 0].sum() <= 1
    # an empty edge list
    got, n = select_dev(L, np.zeros(0, np.float32), np.zeros(0, np.uint64), 1.0, R, cuda, cap=16)
    assert n == 0 and got.size == 0


def test_apply_regions_matches_the_oracle(L, cuda):
    rng = np.random.default_rng(9)
    R, C = 20000, 4
    g = random_stats(rng, R, C, 10, extremes=False)
    alive = rng.random(R) < 0.8
    a = rng.integers(0, R, 8000)
    b = rng.integers(0, R, 8000)
    ok = alive[a] & alive[b]
    root = o.min_root_propagate(R, a[ok], b[ok])
    root = np.where(alive, root, np.arange(R))                  # dead regions point at themselves here
    moved = alive & (root != np.arange(R))
    area, perim = g["area"].copy(), g["perim"].copy()
    bsum, bsq, box = g["bsum"].copy(), g["bsq"].copy(), g["bbox"].copy()
    np.add.at(area, root[moved], g["area"][moved])
    np.add.at(perim, root[moved], g["perim"][moved])
    np.add.at(bsum, root[moved], g["bsum"][moved])
    np.add.at(bsq, root[moved], g["bsq"][moved])
    np.minimum.at(box[:, 0], root[moved], g["bbox"][moved, 0])
    np.minimum.at(box[:, 1], root[moved], g["bbox"][moved, 1])
    np.maximum.at(box[:, 2], root[moved], g["bbox"][moved, 2])
    np.maximum.at(box[:, 3], root[moved], g["bbox"][moved, 3])
    changed = np.zeros(R, bool)
    changed[root[moved]] = True
    d = dict(parent=T(root.astype(np.int32), cuda), alive=T(alive.astype(np.uint8), cuda),
             changed=T(rng.integers(0, 2, R).astype(np.uint8), cuda), area=I64(g["area"], cuda), perim=I64(g["perim"], cuda),
             bsum=I64(g["bsum"], cuda), bsq=I64(g["bsq"], cuda), box=T(g["bbox"], cuda),
             n=torch.full((1,), -1, dtype=torch.int64, device=cuda))
    L.check(L.dm_merge_apply_regions(*[d[k].data_ptr() for k in ("parent", "alive", "changed", "area", "perim", "bsum", "bsq")],
                                     C, d["box"].data_ptr(), R, d["n"].data_ptr(), stream()), "dm_merge_apply_regions")
    assert int(d["n"].item()) == int(moved.sum()) > 1000
    assert np.array_equal(d["alive"].cpu().numpy().astype(bool), alive & ~moved)
    assert np.array_equal(d["changed"].cpu().numpy().astype(bool), changed)
    assert np.array_equal(d["area"].cpu().numpy(), area) and np.array_equal(d["perim"].cpu().numpy(), perim)
    assert np.array_equal(u64(d["bsum"]), bsum) and np.array_equal(u64(d["bsq"]), bsq)
    assert np.array_equal(d["box"].cpu().numpy(), box)


# ------------------------------------------------------------------------------------------
# the whole loop
# ------------------------------------------------------------------------------------------
def assert_same_run(got, want, labels_want):
    assert got.rounds == want["rounds"] and got.merges == want["merges"]
    assert np.array_equal(got.root.cpu().numpy(), want["root"])
    assert np.array_equal(got.area.cpu().numpy(), want["area"]) and np.array_equal(got.perimeter.cpu().numpy(), want["perim"])
    assert np.array_equal(u64(got.band_sum), want["bsum"]) and np.array_equal(u64(got.band_sumsq), want["bsq"])
    assert np.array_equal(got.bbox.cpu().numpy(), want["bbox"])
    assert np.array_equal(u64(got.edge_keys), want["keys"])
    assert np.array_equal(got.boundary_len.cpu().numpy().view(np.uint32), want["blen"])
    assert np.array_equal(bits(got.scores), bits(want["scores"]))
    assert np.array_equal(got.labels.cpu().numpy(), labels_want)


SCENES = [  # H, W, R, C, scale, shape, compactness, nodata, host inputs
    (256, 256, 400, 4, 30.0, 0.1, 0.5, False, True),
    (512, 384, 1200, 3, 40.0, 0.5, 0.2, True, False),
    (1024, 1024, 6000, 1, 25.0, 0.3, 0.8, False, False),
    (2048, 2048, 25000, 4, 50.0, 0.1, 0.5, True, True),
]


@pytest.mark.parametrize("H,W,R,C,scale,shape,cmpct,nodata,host", SCENES)
def test_merge_scene_spectral_bit_exact(cuda, H, W, R, C, scale, shape, cmpct, nodata, host):
    from deepmerge_b200 import merge_scene_spectral
    sc = o.synth_scene(H, W, R, C=C, P=1, D=1, seed=77 + C)
    lab, img, n = sc["labels"].copy(), sc["image"], sc["n_regions"]
    if nodata:
        lab[H // 5: H // 3, W // 4: W // 2] = -1
        lab[:, -3:] = -1
    want = so.merge_scene_spectral(lab, img, n, scale, shape, cmpct)
    assert want["rounds"] > 2 and want["merges"] > n // 4
    got = merge_scene_spectral(lab if host else T(lab, cuda), img if host else T(img, cuda), n_regions=n, scale=scale,
                               shape=shape, compactness=cmpct)
    assert got.labels.is_cuda != host
    assert_same_run(got, want, want["labels"])


def test_band_weights_and_max_rounds(cuda):
    from deepmerge_b200 import merge_scene_spectral
    sc = o.synth_scene(384, 512, 1500, C=4, P=1, D=1)
    bw = [0.5, 2.0, 0.0, 1.25]
    for max_rounds in (0, 2, None):
        want = so.merge_scene_spectral(sc["labels"], sc["image"], sc["n_regions"], 35.0, 0.2, 0.5, bw, max_rounds)
        got = merge_scene_spectral(T(sc["labels"], cuda), T(sc["image"], cuda), n_regions=sc["n_regions"], scale=35.0,
                                   shape=0.2, band_weights=bw, max_rounds=max_rounds)
        assert_same_run(got, want, want["labels"])


def test_full_size_configs1_against_the_oracles(cuda):
    """configs[1] itself: 10k x 10k, 4 bands, ~98k regions; the raster stages by the C oracle, the loop by numpy."""
    from deepmerge_b200 import MergeEngine
    from deepmerge_b200.synth import synth_scene
    from oracle import build as oc
    Hf = Wf = 10000
    sc = synth_scene(Hf, Wf, 100000, C=4, device=cuda)
    R = sc.n_regions
    lab, img = sc.labels.cpu().numpy(), sc.image.cpu().numpy()
    k, b, area, per = oc.build_rag(lab, R)
    s, q = oc.pool_bands(lab, img, R)
    box = o.region_bbox(lab, R)
    del img
    want = so.merge_spectral(area, per, s, q, box, k, b, np.float32(60.0 * 60.0), 0.1, 0.5)
    eng = MergeEngine(Hf, Wf, R, 0, C=4, n_points=0, device=cuda)
    got = eng.run_spectral(sc.labels, sc.image, 60.0)
    assert want["rounds"] > 2 and want["merges"] > R // 2
    assert_same_run(got, want, oc.relabel(lab, want["root"]))


def test_determinism_and_shared_buffers_with_the_l2_loop(cuda):
    """Two spectral runs on one engine are bit-equal (the second replays the captured round graphs), and the L2 loop on
    the same engine equals its oracle before and after them.  The round graph is captured once per criterion and
    parameters: runs that repeat them replay it."""
    from deepmerge_b200 import MergeEngine
    sc = o.synth_scene(512, 640, 2000, C=4)
    n = sc["n_regions"]
    d = {k: T(sc[k], cuda) for k in ("labels", "image", "feats", "xs", "ys")}
    eng = MergeEngine(512, 640, n, sc["feats"].shape[1], C=4, n_points=sc["feats"].shape[0], device=cuda)
    l2 = o.merge_scene(sc["labels"], n, sc["region_of_point"], sc["feats"], tau=0.5)

    def run_l2():
        r = eng.run(d["labels"], d["feats"], 0.5, image=d["image"], xs=d["xs"], ys=d["ys"])
        assert r.rounds == l2["rounds"] and r.merges == l2["merges"]
        assert np.array_equal(r.labels.cpu().numpy(), l2["labels"]) and np.array_equal(u64(r.edge_keys), l2["keys"])

    run_l2()
    run_l2()
    assert l2["rounds"] >= 1 and len(eng._graphs) == 1
    want = so.merge_scene_spectral(sc["labels"], sc["image"], n, 30.0)
    runs = []
    for _ in range(2):
        r = eng.run_spectral(d["labels"], d["image"], 30.0)
        assert_same_run(r, want, want["labels"])
        runs.append((r.labels.clone(), r.scores.clone(), r.root.clone()))
    assert all(torch.equal(x, y) for x, y in zip(*runs))
    assert want["rounds"] > 2 and eng.use_graphs and len(eng._graphs) == 2
    run_l2()
    assert len(eng._graphs) == 2


def test_quality_on_the_synthetic_scene(cuda):
    """Region colour = object colour +- 4, pixel noise +- 8: with shape = 0 and scale 50 (chosen with the CPU oracle: the
    largest round value that keeps every segment within one object on these scenes) no merged segment covers pixels of
    two ground-truth objects, and the segments left are what the oracle leaves."""
    from deepmerge_b200 import merge_scene_spectral
    sc = o.synth_scene(1024, 1024, 6000, C=4, P=1, D=1)
    n, obj = sc["n_regions"], sc["region_obj"]
    got = merge_scene_spectral(T(sc["labels"], cuda), T(sc["image"], cuda), n_regions=n, scale=50.0, shape=0.0)
    root = got.root.cpu().numpy()
    lo = np.full(n, np.iinfo(np.int32).max)
    hi = np.full(n, -1)
    np.minimum.at(lo, root, obj)
    np.maximum.at(hi, root, obj)
    assert not ((hi >= 0) & (lo != hi)).any(), "a segment covers two objects"
    left = len(np.unique(root))
    want = so.merge_scene_spectral(sc["labels"], sc["image"], n, 50.0, 0.0)
    print("segments left: %d of %d regions, %d objects" % (left, n, sc["n_objects"]))
    assert left == len(np.unique(want["root"])) and sc["n_objects"] <= left < n // 10
