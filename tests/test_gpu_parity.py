"""GPU parity: the CUDA path (through the C ABI) against the CPU oracle on the same seeded
inputs.  Bit-exact for integer / index work (edge sets, counts, label maps, band sums,
pooled means with reference summation order); stated tolerances for fp32 scores."""
import ctypes
import os

import numpy as np
import pytest

from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


def T(x, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def keys_np(t):
    return t.cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------------------------------
# primitives
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,R", [(0, 10), (1, 2), (777, 5), (5000, 70000), (300000, 1 << 20), (70000, 3), (2500000, 1 << 14)])
def test_sort_edges(cuda, n, R):
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(n + R)
    lo = rng.integers(0, R, n)
    hi = rng.integers(0, R, n)
    keys = (lo.astype(np.uint64) << np.uint64(32)) | hi.astype(np.uint64)
    vals = np.arange(n, dtype=np.uint32)
    cap = n + 100
    k = torch.zeros(cap, dtype=torch.int64, device=cuda)
    v = torch.zeros(cap, dtype=torch.int32, device=cuda)
    k[:n] = T(keys.view(np.int64), cuda)
    v[:n] = T(vals.view(np.int32), cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    wsb = L.dm_sort_edges_workspace_bytes(cap)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
    L.check(L.dm_sort_edges(k.data_ptr(), v.data_ptr(), nd.data_ptr(), cap, R, ws.data_ptr(), wsb, None), "sort")
    torch.cuda.synchronize()
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(keys_np(k[:n]), keys[order])
    assert np.array_equal(v[:n].cpu().numpy().view(np.uint32), vals[order])      # stable


@pytest.mark.parametrize("n,R", [(0, 10), (1, 2), (2048, 3), (5000, 40), (300000, 700), (2500000, 2500), (20000, 100),
                                 (600000, 200000), (3000000, 6000)])
def test_edges_sort_unique(cuda, n, R):
    """Run reduction of an edge list (one cooperative launch when available): unique keys ascending, lengths summed.
    The cases cover the hashed path with small buckets, with hub buckets (R = 100, 700), and its fall-back to the radix
    sort because more buckets are hubs than the hub list holds (R = 2500 and R = 6000; the largest bucket of R = 6000
    holds 544 unique keys, far below the hub limit).  tests/test_gpu_prims_exact.py covers every path at its
    thresholds."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(7 * n + R)
    lo = rng.integers(0, R, n)
    hi = rng.integers(0, R, n)
    keys = (lo.astype(np.uint64) << np.uint64(32)) | hi.astype(np.uint64)
    lens = rng.integers(1, 1000, n).astype(np.uint32)
    cap = n + 33
    k = torch.full((cap,), -1, dtype=torch.int64, device=cuda)
    v = torch.full((cap,), 12345, dtype=torch.int32, device=cuda)
    k[:n] = T(keys.view(np.int64), cuda)
    v[:n] = T(lens.view(np.int32), cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    nout = torch.full((1,), -1, dtype=torch.int64, device=cuda)
    wsb = L.dm_edges_unique_workspace_bytes(cap)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
    L.check(L.dm_edges_sort_unique(k.data_ptr(), v.data_ptr(), nd.data_ptr(), cap, R, nout.data_ptr(), ws.data_ptr(), wsb,
                                   None), "sort_unique")
    torch.cuda.synchronize()
    uk, inv = np.unique(keys, return_inverse=True)
    want = np.bincount(inv, weights=lens.astype(np.float64), minlength=len(uk)).astype(np.uint64)
    m = int(nout.item())
    assert m == len(uk)
    assert np.array_equal(keys_np(k[:m]), uk)
    assert np.array_equal(v[:m].cpu().numpy().view(np.uint32).astype(np.uint64), want)


@pytest.mark.parametrize("n", [0, 1, 2047, 2048, 2049, 100000, 3000000])
def test_scan(cuda, n):
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(n)
    x = rng.integers(0, 5, n).astype(np.uint32)
    cap = n + 5
    xin = torch.zeros(cap, dtype=torch.int32, device=cuda)
    xin[:n] = T(x.view(np.int32), cuda)
    out = torch.zeros(cap, dtype=torch.int32, device=cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    tot = torch.full((1,), -1, dtype=torch.int64, device=cuda)
    wsb = L.dm_scan_workspace_bytes(cap)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
    L.check(L.dm_scan_exclusive_u32(xin.data_ptr(), out.data_ptr(), nd.data_ptr(), cap, tot.data_ptr(), ws.data_ptr(), wsb,
                                    None), "scan")
    ex = np.cumsum(x, dtype=np.int64) - x
    assert np.array_equal(out[:n].cpu().numpy().view(np.uint32), ex.astype(np.uint32))
    assert int(tot.item()) == int(x.sum())


@pytest.mark.parametrize("R,N,hub", [(500, 3000, 0), (200_000, 1_000, 0), (100, 20_000, 5_000)])
def test_csr_build_matches_oracle(cuda, R, N, hub):
    """Region -> point CSR (bucket sort with offsets) against the oracle.  The cases: random regions with invalid points;
    many more regions than points (per-id arrays sized from the region count); one region holding `hub` points, above
    the bucket sort's hub limit, so the radix path inside the same launch and its binary-search offsets run."""
    from deepmerge_b200 import csr_from_region_of_point
    rng = np.random.default_rng(R + N)
    rop = rng.integers(-1, R, N).astype(np.int32)
    rop[rng.choice(N, hub, replace=False)] = R // 2
    off, ids = csr_from_region_of_point(T(rop, cuda), R)
    ho, hi = o.csr_from_region_of_point(rop, R)
    assert np.array_equal(off.cpu().numpy(), ho)
    assert np.array_equal(ids.cpu().numpy()[: hi.size], hi)


# ------------------------------------------------------------------------------------------
# synthetic generator: device == oracle, bit for bit
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,R,C", [(96, 130, 40, 3), (257, 300, 500, 4), (64, 64, 4096, 1)])
def test_synth_matches_oracle(cuda, H, W, R, C):
    from deepmerge_b200.synth import synth_scene
    d = synth_scene(H, W, R, C=C, device=cuda)
    h = o.synth_scene(H, W, R, C=C)
    assert d.n_regions == h["n_regions"]
    assert np.array_equal(d.labels.cpu().numpy(), h["labels"])
    assert np.array_equal(d.region_obj.cpu().numpy(), h["region_obj"])
    assert np.array_equal(d.image.cpu().numpy(), h["image"])
    assert np.array_equal(d.xs.cpu().numpy(), h["xs"]) and np.array_equal(d.ys.cpu().numpy(), h["ys"])
    assert np.array_equal(d.region_of_point.cpu().numpy(), h["region_of_point"])
    assert np.array_equal(d.feats.cpu().numpy(), h["feats"])


# ------------------------------------------------------------------------------------------
# R1 RAG (+ fused band pooling)
# ------------------------------------------------------------------------------------------
def check_rag(cuda, L, R, image=None, labels_dev=None, **kw):
    """build_rag on labels_dev (default: a contiguous device copy of L) against the oracle on L."""
    from deepmerge_b200 import build_rag
    rag = build_rag(T(L, cuda) if labels_dev is None else labels_dev, R, None if image is None else T(image, cuda), **kw)
    okw = {}
    if "rows_own" in kw:
        okw = dict(own_rows=kw["rows_own"], top_border=kw.get("top_border", True), bottom_border=kw.get("bottom_border", True))
    keys, blen, area, per = o.build_rag(L, R, **okw)
    assert np.array_equal(keys_np(rag.edge_keys), keys)
    assert np.array_equal(rag.boundary_len.cpu().numpy().view(np.uint32), blen)
    assert np.array_equal(rag.area.cpu().numpy(), area)
    assert np.array_equal(rag.perimeter.cpu().numpy(), per)
    if image is not None:
        own = kw.get("rows_own", L.shape[0])
        s, q = o.pool_bands(L[:own], image[:own], R)
        assert np.array_equal(rag.band_sum.cpu().numpy().view(np.uint64), s)
        assert np.array_equal(rag.band_sumsq.cpu().numpy().view(np.uint64), q)
    return rag


@pytest.mark.parametrize("H,W", [(1, 1), (1, 7), (5, 1), (33, 128), (32, 256), (33, 257), (64, 260), (100, 1000),
                                 (65, 516), (300, 1024)])
@pytest.mark.parametrize("C", [0, 4])
def test_rag_random_rasters(cuda, H, W, C):
    rng = np.random.default_rng(H * 1000 + W + C)
    R = 37
    small = rng.integers(0, R, size=((H + 5) // 6, (W + 6) // 7)).astype(np.int32)
    L = np.kron(small, np.ones((6, 7), np.int32))[:H, :W].copy()
    L[rng.random((H, W)) < 0.02] = rng.integers(0, R)            # speckle
    img = rng.integers(0, 256, size=(H, W, C)).astype(np.uint8) if C else None
    check_rag(cuda, L, R, img)


@pytest.mark.parametrize("C", [1, 2, 3, 4])
def test_rag_bands_all_channel_counts(cuda, C):
    sc = o.synth_scene(150, 512, 300, C=C)
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])


def test_rag_nodata_and_every_pixel_its_own_region(cuda):
    rng = np.random.default_rng(5)
    H, W = 70, 300
    L = rng.integers(0, 50, size=(H, W)).astype(np.int32)         # pure noise: ~every pair is an edge
    L[rng.random((H, W)) < 0.1] = -1
    L[10:20, 40:90] = -1
    img = rng.integers(0, 256, size=(H, W, 4)).astype(np.uint8)
    check_rag(cuda, L, 50, img)
    L2 = np.arange(H * W, dtype=np.int32).reshape(H, W)           # E = 2HW - H - W, tables saturate
    check_rag(cuda, L2, H * W, img, capacity=2 * H * W)


@pytest.mark.parametrize("islands", [300, 5000])
@pytest.mark.parametrize("background_first", [True, False])
def test_rag_hub_region(cuda, islands, background_first):
    """One background region touching hundreds / thousands of islands: a bucket of the hashed run reduction that is
    ranked by a whole block (300) or sends the call down the radix path (5000, when the background has the lowest id)."""
    side = int(np.ceil(np.sqrt(islands)))
    H = W = 4 * side + 3
    bg = 0 if background_first else islands
    L = np.full((H, W), bg, np.int32)
    k = 0
    for i in range(side):
        for j in range(side):
            if k < islands:
                L[4 * i + 2:4 * i + 4, 4 * j + 2:4 * j + 5] = k + (1 if background_first else 0)
                k += 1
    rag = check_rag(cuda, L, islands + 1)
    assert rag.n_edges >= islands


def test_rag_capacity_overflow_is_reported_and_retried(cuda):
    L = np.arange(64 * 256, dtype=np.int32).reshape(64, 256)
    from deepmerge_b200 import build_rag
    rag = build_rag(T(L, cuda), 64 * 256, capacity=1000)          # too small on purpose
    keys, blen, area, per = o.build_rag(L, 64 * 256)
    assert np.array_equal(keys_np(rag.edge_keys), keys)


def test_rag_label_out_of_range_raises(cuda):
    from deepmerge_b200 import build_rag
    L = np.zeros((40, 40), np.int32)
    L[3, 3] = 99
    with pytest.raises(ValueError):
        build_rag(T(L, cuda), 10)


def test_rag_strided_and_unaligned_rasters_take_fallback_path(cuda):
    import torch
    sc = o.synth_scene(90, 301, 120, C=3)                         # W*C not a multiple of 4, ld odd
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])
    big = T(o.synth_scene(90, 320, 120, C=4)["labels"], cuda)
    from deepmerge_b200 import build_rag
    view = big[:, 3:300]                                          # pitch 320, base misaligned
    rag = build_rag(view, 200)
    keys, blen, area, per = o.build_rag(view.cpu().numpy(), 200)
    assert np.array_equal(keys_np(rag.edge_keys), keys) and np.array_equal(rag.perimeter.cpu().numpy(), per)


def test_rag_forced_fallback_equals_tma(cuda):
    """One raster through both staging paths: TMA for the aligned copy, ld.global for a copy whose base is 4 bytes off
    16-byte alignment (pitch still aligned)."""
    from deepmerge_b200._lib import lib
    sc = o.synth_scene(130, 512, 400, C=4)
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])
    assert lib().dm_rag_last_path() == 1
    wide = T(np.zeros((130, 516), np.int32), cuda)
    view = wide[:, 1:513]
    view.copy_(T(sc["labels"], cuda))
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"], labels_dev=view)
    assert lib().dm_rag_last_path() == 0


def test_rag_alternative_kernel_shapes(cuda):
    """4-band rasters of three shapes; long strips wrap the item buffers."""
    sc = o.synth_scene(300, 1024, 350, C=4)
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])
    rng = np.random.default_rng(3)
    L = rng.integers(0, 50, size=(70, 300)).astype(np.int32)
    L[rng.random(L.shape) < 0.1] = -1
    check_rag(cuda, L, 50, rng.integers(0, 256, size=(70, 300, 4)).astype(np.uint8))
    sc = o.synth_scene(3000, 2048, 24000, C=4)        # long strips: the item buffers / the ring wrap around many times
    check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])


def test_rag_row_tiles_sum_to_whole(cuda):
    from deepmerge_b200 import build_rag, merge_edge_lists
    import torch
    sc = o.synth_scene(260, 384, 500, C=4)
    L, R, img = sc["labels"], sc["n_regions"], sc["image"]
    whole = check_rag(cuda, L, R, img)
    cuts = [0, 64, 65, 170, 260]
    ks, bs, area, border, bsum = [], [], 0, 0, 0
    for i in range(len(cuts) - 1):
        y0, y1 = cuts[i], cuts[i + 1]
        last = y1 == 260
        tile = L[y0:y1 + (0 if last else 1)]
        r = check_rag(cuda, tile, R, img[y0:y1 + (0 if last else 1)], rows_own=y1 - y0, top_border=y0 == 0,
                      bottom_border=last)
        ks.append(r.edge_keys); bs.append(r.boundary_len)
        area = area + r.area; border = border + r.border; bsum = bsum + r.band_sum
    k, b = merge_edge_lists(torch.cat(ks), torch.cat(bs), R)
    assert torch.equal(k, whole.edge_keys) and torch.equal(b, whole.boundary_len)
    assert torch.equal(area, whole.area) and torch.equal(border, whole.border) and torch.equal(bsum, whole.band_sum)


def test_rag_fragmentation_extremes(cuda):
    for R in (6, 40000):                                          # few huge regions / 8-px regions
        sc = o.synth_scene(384, 768, R, C=4)
        check_rag(cuda, sc["labels"], sc["n_regions"], sc["image"])


# ------------------------------------------------------------------------------------------
# R3-R5 pooling
# ------------------------------------------------------------------------------------------
def test_pool_points_bit_exact_with_reference_golden(cuda, golden_dir):
    from deepmerge_b200 import pool_points_csr, region_mean
    p = np.load(os.path.join(golden_dir, "pool_score.npz"))
    off, ids = o.membership_csr(list(p["fields"]))
    s, c = pool_points_csr(T(off, cuda), T(ids, cuda), T(p["store"], cuda))
    mean, _ = region_mean(s, c)
    u = p["used"]
    assert np.array_equal(mean.cpu().numpy()[u], p["means"][u])    # == the reference's np.mean, bit for bit


@pytest.mark.parametrize("D", [1, 31, 100, 128, 200, 300])
def test_pool_points_matches_oracle(cuda, D):
    from deepmerge_b200 import csr_from_region_of_point, pool_points_csr, region_mean
    rng = np.random.default_rng(D)
    R, N = 500, 3000
    rop = rng.integers(-1, R, N).astype(np.int32)
    rop[rop == 7] = 8                                              # an empty region
    feats = rng.standard_normal((N, D)).astype(np.float32)
    off, ids = csr_from_region_of_point(T(rop, cuda), R)
    ho, hi = o.csr_from_region_of_point(rop, R)
    assert np.array_equal(off.cpu().numpy(), ho)
    assert np.array_equal(ids.cpu().numpy()[: hi.size], hi)
    s, c = pool_points_csr(off, ids, T(feats, cuda))
    hs, hc, hm = o.pool_points_csr(ho, hi, feats)
    assert np.array_equal(s.cpu().numpy(), hs) and np.array_equal(c.cpu().numpy(), hc)
    mean, n2 = region_mean(s, c)
    hm = o.region_mean(hs, hc)                                  # NaN rows for regions without points, as np.mean gives
    assert (hc == 0).any() and np.isnan(hm[hc == 0]).all()
    assert np.array_equal(mean.cpu().numpy(), hm, equal_nan=True)
    np.testing.assert_allclose(n2.cpu().numpy(), np.sum(hm.astype(np.float64) ** 2, 1), rtol=1e-5)


def test_points_region_and_pool_dense(cuda):
    import torch
    from deepmerge_b200 import points_region, pool_dense
    sc = o.synth_scene(120, 200, 150, C=1)
    L, R = sc["labels"].copy(), sc["n_regions"]
    L[5:9, 5:40] = -1
    xs = np.r_[sc["xs"], -1, 200, 6].astype(np.int32)
    ys = np.r_[sc["ys"], 3, 3, 6].astype(np.int32)
    rop = points_region(T(L, cuda), T(xs, cuda), T(ys, cuda)).cpu().numpy()
    want = np.where((xs >= 0) & (xs < 200), L[np.clip(ys, 0, 119), np.clip(xs, 0, 199)], -1)
    assert np.array_equal(rop, np.where(want < 0, -1, want))
    rng = np.random.default_rng(0)
    emb = rng.standard_normal((120, 200, 20)).astype(np.float32)
    s, c = pool_dense(T(L, cuda), T(emb, cuda), R)
    hs, hc = o.pool_dense(L, emb, R)
    assert np.array_equal(c.cpu().numpy(), hc)
    np.testing.assert_allclose(s.cpu().numpy(), hs, rtol=1e-3, atol=1e-3)     # fp32 atomics vs float64
    sb, cb = pool_dense(T(L, cuda), T(emb, cuda).to(torch.bfloat16), R)
    hb, _ = o.pool_dense(L, o.bf16_round(emb), R)
    np.testing.assert_allclose(sb.cpu().numpy(), hb, rtol=1e-3, atol=1e-3)


# ------------------------------------------------------------------------------------------
# R6 score
# ------------------------------------------------------------------------------------------
def test_score_l2_against_reference_golden(cuda, golden_dir):
    from deepmerge_b200 import score_l2
    e = np.load(os.path.join(golden_dir, "euclid.npz"))
    K = e["X"].shape[0]
    mean = np.concatenate([e["X"], e["Y"]])
    keys = o.pack_keys(np.arange(K), np.arange(K) + K)
    s = score_l2(T(mean, cuda), T(keys.view(np.int64), cuda)).cpu().numpy()
    tol = o.l2_abs_tolerance(mean, keys)                           # 1e-3 relative + cancellation floor
    assert np.all(np.abs(s - o.score_l2_f64(mean, keys)) <= tol)
    big = e["d"] > 1e-2 * np.sqrt(np.sum(mean[:K] ** 2, 1))        # away from cancellation: 1e-3 relative to the reference
    assert np.all(np.abs(s[big] - e["d"][big]) <= 1e-3 * e["d"][big])


def test_score_l2_synthetic_scene(cuda):
    from deepmerge_b200 import build_rag, pool_points, region_mean, score_l2
    sc = o.synth_scene(300, 300, 900, C=1)
    R = sc["n_regions"]
    keys, *_ = o.build_rag(sc["labels"], R)
    off, ids = o.csr_from_region_of_point(sc["region_of_point"], R)
    _, _, hm = o.pool_points_csr(off, ids, sc["feats"])
    s, c = pool_points(T(sc["region_of_point"], cuda), T(sc["feats"], cuda), R)
    mean, n2 = region_mean(s, c)
    got = score_l2(mean, T(keys.view(np.int64), cuda), n2).cpu().numpy()
    assert np.all(np.abs(got - o.score_l2_f64(hm, keys)) <= o.l2_abs_tolerance(hm, keys))


# ------------------------------------------------------------------------------------------
# R9 merge loop + relabel
# ------------------------------------------------------------------------------------------
def random_graph(seed, R=300, E=900, D=16):
    rng = np.random.default_rng(seed)
    u = rng.integers(0, R, E)
    v = (u + rng.integers(1, R, E)) % R
    keys, inv = np.unique(o.pack_keys(u, v), return_inverse=True)
    blen = rng.integers(1, 50, keys.size).astype(np.uint32)
    cluster = rng.integers(0, 12, R)
    centres = rng.standard_normal((12, D)).astype(np.float32) * 0.6
    cnt = rng.integers(0, 6, R).astype(np.int32)
    # integer-valued sums on a coarse grid keep every fp32 sum exact, so decisions cannot
    # depend on summation order even though clusters are close (multi-round merges happen)
    mean = np.round((centres[cluster] + 0.05 * rng.standard_normal((R, D))) * 64) / 64
    sum_ = (mean * np.maximum(cnt, 1)[:, None]).astype(np.float32)
    sum_[cnt == 0] = 0
    area = rng.integers(1, 1000, R).astype(np.int64)
    per = (rng.integers(1, 100, R) + 2000).astype(np.int64)
    return sum_, cnt, area, per, keys, blen


# D = 16 runs the vec L2 kernel in one trip, D = 7 the scalar kernel, D = 260 the vec kernel in three trips
@pytest.mark.parametrize("seed,tau,D", [pytest.param(seed, tau, D, id="%s-%d%s" % (tau, seed, "" if D == 16 else "-D%d" % D))
                                        for D in (16, 7, 260) for tau in (0.5, 1.5, 3.0) for seed in range(5)])
def test_merge_graph_matches_oracle(cuda, seed, tau, D):
    from deepmerge_b200 import merge_graph
    sum_, cnt, area, per, keys, blen = random_graph(seed, D=D)
    want = o.merge_graph(sum_, cnt, area, per, keys, blen, tau=tau)
    got = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(per, cuda), T(keys.view(np.int64), cuda),
                      T(blen.view(np.int32), cuda), tau)
    assert np.array_equal(got.root.cpu().numpy(), want["root"])
    assert got.rounds == want["rounds"] and got.merges == want["merges"]
    assert np.array_equal(keys_np(got.edge_keys), want["keys"])
    assert np.array_equal(got.boundary_len.cpu().numpy().view(np.uint32), want["blen"])
    roots = np.unique(want["root"])
    assert np.array_equal(got.area.cpu().numpy()[roots], want["area"][roots])
    assert np.array_equal(got.perimeter.cpu().numpy()[roots], want["perim"][roots])
    assert np.array_equal(got.cnt.cpu().numpy()[roots], want["cnt"][roots])
    assert np.array_equal(got.sum.cpu().numpy()[roots], want["sum"][roots])       # fixed summation order
    np.testing.assert_allclose(got.scores.cpu().numpy(), want["scores"], rtol=1e-3, atol=1e-3)


def test_regions_without_sample_points_never_merge(cuda):
    """A region without points has no embedding (np.mean over no rows is NaN, ExtractFeatures.py:211):
    its edges score NaN and are never selected -- neither against another empty region (a made-up zero vector would
    score 0) nor against a low-norm neighbour -- for the L2 scorer and for the pair-MLP."""
    from deepmerge_b200 import PackedMLP, merge_graph
    R, D = 6, 4
    #   0 -- 1 -- 2 -- 3 -- 4 -- 5      1 and 2 are empty, 3 has a tiny embedding, 4 / 5 are close to each other
    keys = o.pack_keys(np.arange(R - 1), np.arange(1, R))
    blen = np.ones(R - 1, np.uint32)
    cnt = np.array([2, 0, 0, 1, 1, 1], np.int32)
    sum_ = np.zeros((R, D), np.float32)
    sum_[0] = 6.0
    sum_[3] = 1e-3
    sum_[4] = 5.0
    sum_[5] = 5.01
    area = np.full(R, 10, np.int64)
    per = np.full(R, 14, np.int64)
    want = o.merge_graph(sum_, cnt, area, per, keys, blen, tau=0.5)
    assert want["merges"] == 1 and np.array_equal(want["root"], [0, 1, 2, 3, 4, 4])       # only 4 -- 5
    got = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(per, cuda), T(keys.view(np.int64), cuda),
                      T(blen.view(np.int32), cuda), 0.5)
    assert np.array_equal(got.root.cpu().numpy(), want["root"]) and got.merges == 1
    sc = got.scores.cpu().numpy()
    assert np.isnan(sc[:3]).all() and np.isfinite(sc[3:]).all()                           # edges 0-1, 1-2, 2-3 have no score
    # the same with a pair-MLP that says "merge" for EVERY finite input
    h = 2 * D
    Wm = [np.zeros((h, 2 * D), np.float32), np.zeros(h, np.float32), np.zeros((h, h), np.float32), np.zeros(h, np.float32),
          np.zeros((2, h), np.float32), np.array([0.0, 1.0], np.float32)]
    want = o.merge_graph(sum_, cnt, area, per, keys, blen, mlp=tuple(Wm), mlp_bf16=True, max_rounds=1)
    got = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(per, cuda), T(keys.view(np.int64), cuda),
                      T(blen.view(np.int32), cuda), 0.0, mlp=PackedMLP(*[T(w, cuda) for w in Wm]), max_rounds=1)
    assert np.array_equal(want["root"], [0, 1, 2, 3, 3, 3])                               # 3 -- 4 -- 5 only
    assert np.array_equal(got.root.cpu().numpy(), want["root"])


def test_cascade_scene_needs_three_rounds_and_equals_the_oracle(cuda):
    """The multi-round workload of bench.py: the device generator equals the oracle's, the merge takes exactly three
    rounds (regions -> objects -> groups -> tops), and roots / label map / merged statistics equal the oracle's after
    every round limit."""
    from deepmerge_b200 import merge_scene
    from deepmerge_b200.synth import CASCADE_TAU, cascade_feats, synth_scene
    H, W, R = 600, 800, 4000
    sc = o.synth_scene(H, W, R, C=4)
    d = synth_scene(H, W, R, C=4, device=cuda)
    f = o.synth_cascade_feats(sc["region_of_point"], sc["region_obj"], H, W, R)
    fd = cascade_feats(d)
    assert np.array_equal(fd.cpu().numpy(), f)
    n = sc["n_regions"]
    for mr in (1, 2, 64):
        want = o.merge_scene(sc["labels"], n, sc["region_of_point"], f, tau=CASCADE_TAU, max_rounds=mr)
        got = merge_scene(d.labels, fd, CASCADE_TAU, n_regions=n, image=d.image, xs=d.xs, ys=d.ys, max_rounds=mr)
        assert got.rounds == want["rounds"] == min(mr, 3) and got.merges == want["merges"]
        assert np.array_equal(got.root.cpu().numpy(), want["root"])
        assert np.array_equal(got.labels.cpu().numpy(), want["labels"])
        roots = np.unique(want["root"])
        assert np.array_equal(got.area.cpu().numpy()[roots], want["area"][roots])
        assert np.array_equal(got.perimeter.cpu().numpy()[roots], want["perim"][roots])
        assert np.array_equal(keys_np(got.edge_keys), want["keys"])


def test_merge_graph_max_rounds_and_snake(cuda):
    from deepmerge_b200 import merge_graph
    R, D = 5000, 8
    keys = o.pack_keys(np.arange(R - 1), np.arange(1, R))          # one long chain: deep union-find trees
    blen = np.ones(R - 1, np.uint32)
    sum_ = np.zeros((R, D), np.float32)
    cnt = np.ones(R, np.int32)
    area = np.ones(R, np.int64)
    per = np.full(R, 4, np.int64)
    got = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(per, cuda), T(keys.view(np.int64), cuda),
                      T(blen.view(np.int32), cuda), 0.5)
    assert np.all(got.root.cpu().numpy() == 0) and got.rounds == 1 and got.merges == R - 1
    assert int(got.area[0]) == R and int(got.perimeter[0]) == 4 * R - 2 * (R - 1) and got.edge_keys.shape[0] == 0
    none = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(per, cuda), T(keys.view(np.int64), cuda),
                       T(blen.view(np.int32), cuda), 0.5, max_rounds=0)
    assert none.rounds == 0 and np.array_equal(none.root.cpu().numpy(), np.arange(R))


@pytest.mark.parametrize("H,W,R,C", [(200, 256, 300, 4), (333, 517, 1500, 3), (64, 64, 10, 0)])
def test_merge_scene_end_to_end_bit_exact(cuda, H, W, R, C):
    from deepmerge_b200 import merge_scene
    sc = o.synth_scene(H, W, R, C=max(C, 1))
    want = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], tau=0.5)
    got = merge_scene(T(sc["labels"], cuda), T(sc["feats"], cuda), 0.5, n_regions=sc["n_regions"],
                      image=T(sc["image"], cuda) if C else None, xs=T(sc["xs"], cuda), ys=T(sc["ys"], cuda))
    assert np.array_equal(got.labels.cpu().numpy(), want["labels"])                 # final label map, bit exact
    assert np.array_equal(got.root.cpu().numpy(), want["root"])
    assert got.rounds == want["rounds"] and got.merges == want["merges"]
    # host inputs (numpy) take the same path through pinned staging and come back on the host
    host = merge_scene(sc["labels"], sc["feats"], 0.5, n_regions=sc["n_regions"], image=sc["image"] if C else None,
                       region_of_point=sc["region_of_point"])
    assert not host.labels.is_cuda and np.array_equal(host.labels.numpy(), want["labels"])


def test_relabel_and_compact(cuda):
    from deepmerge_b200 import compact_roots, relabel
    rng = np.random.default_rng(1)
    R = 1000
    root = o.union_find_min_root(R, rng.integers(0, R, 600), rng.integers(0, R, 600)).astype(np.int32)
    for H, W in [(64, 64), (37, 53), (1, 5)]:
        L = rng.integers(-1, R, size=(H, W)).astype(np.int32)
        got = relabel(T(L, cuda), T(root, cuda)).cpu().numpy()
        assert np.array_equal(got, o.relabel(L, root))
    c, n = compact_roots(T(root, cuda))
    hc, hn = o.compact_roots(root)
    assert n == hn and np.array_equal(c.cpu().numpy(), hc)


def test_determinism_run_twice(cuda):
    from deepmerge_b200 import merge_scene
    sc = o.synth_scene(256, 384, 800, C=4)
    args = dict(n_regions=sc["n_regions"], image=T(sc["image"], cuda), xs=T(sc["xs"], cuda), ys=T(sc["ys"], cuda))
    a = merge_scene(T(sc["labels"], cuda), T(sc["feats"], cuda), 0.5, **args)
    la, sa, ka = a.labels.clone(), a.sum.clone(), a.edge_keys.clone()
    b = merge_scene(T(sc["labels"], cuda), T(sc["feats"], cuda), 0.5, **args)
    import torch
    assert torch.equal(la, b.labels) and torch.equal(sa, b.sum) and torch.equal(ka, b.edge_keys)


# ------------------------------------------------------------------------------------------
# empty inputs
# ------------------------------------------------------------------------------------------
def test_empty_inputs(cuda):
    import torch
    from deepmerge_b200 import build_rag, pool_points, relabel
    rag = build_rag(torch.zeros((0, 16), dtype=torch.int32, device=cuda), 4)
    assert rag.n_edges == 0 and int(rag.area.sum()) == 0
    s, c = pool_points(torch.zeros(0, dtype=torch.int32, device=cuda), torch.zeros((0, 8), device=cuda), 3)
    assert int(c.sum()) == 0 and float(s.abs().sum()) == 0
    assert relabel(torch.zeros((0, 4), dtype=torch.int32, device=cuda), torch.zeros(2, dtype=torch.int32, device=cuda)).numel() == 0
    with pytest.raises(ValueError):
        build_rag(torch.zeros((4, 4), dtype=torch.int32), 4)       # CPU tensor: no CPU path


def test_pool_boundary_matches_oracle(cuda):
    """Per-boundary pooling of a dense embedding grid: counts exact (= 2 * boundary_len), sums within 1e-3
    relative of a float64 restatement (fp32 atomics, order not fixed)."""
    import torch
    from deepmerge_b200 import build_rag, pool_boundary
    sc = o.synth_scene(96, 200, 150, C=0)
    L, R = sc["labels"].copy(), sc["n_regions"]
    L[5:9, 20:40] = -1
    rng = np.random.default_rng(3)
    for D, dt in ((100, torch.float32), (24, torch.bfloat16)):
        emb = rng.standard_normal((96, 200, D)).astype(np.float32)
        rag = build_rag(T(L, cuda), R)
        emb_t = T(emb, cuda).to(dt)
        s, c = pool_boundary(T(L, cuda), emb_t, rag.edge_keys)
        ws, wc = o.pool_boundary(L, emb_t.float().cpu().numpy(), keys_np(rag.edge_keys))
        assert np.array_equal(c.cpu().numpy(), wc)
        assert np.array_equal(wc, 2 * rag.boundary_len.cpu().numpy().view(np.uint32).astype(np.int64))
        np.testing.assert_allclose(s.cpu().numpy(), ws, rtol=1e-3, atol=1e-3)


def test_scene_pipeline_equals_single_calls(cuda):
    """ScenePipeline (overlapped H2D / compute / D2H over a stream of host scenes) returns, in order, exactly
    the label maps of one-at-a-time calls."""
    import torch
    from deepmerge_b200 import MergeEngine, ScenePipeline
    scenes, want = [], []
    for seed in (1, 2, 3, 4, 5):
        sc = o.synth_scene(128, 256, 200, C=4, seed=seed)
        R = sc["n_regions"]
        scenes.append({k: torch.from_numpy(np.ascontiguousarray(sc[k])).pin_memory() for k in ("labels", "image", "feats", "xs", "ys")})
        want.append(o.merge_scene(sc["labels"], R, sc["region_of_point"], sc["feats"], tau=0.5)["labels"])
    assert len({o.synth_scene(128, 256, 200, C=4, seed=s)["n_regions"] for s in (1, 2, 3, 4, 5)}) == 1
    eng = MergeEngine(128, 256, R, 100, C=4, n_points=scenes[0]["feats"].shape[0], device=cuda)
    got = [lab.clone().numpy() for lab in ScenePipeline(eng).run(iter(scenes), 0.5)]
    assert len(got) == 5
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


def test_rag_against_c_oracle_at_medium_size(cuda):
    """3000 x 4096, 12k regions, 4 bands, nodata holes: bit-exact against the plain-C restatement (fast enough for this
    size) and the whole merge against a recount of the merged map by the same C code."""
    from deepmerge_b200 import build_rag, merge_scene
    from oracle import build as oc
    sc = o.synth_scene(3000, 4096, 12000, C=4)
    L, R = sc["labels"].copy(), sc["n_regions"]
    L[100:140, 900:1500] = -1
    L[2990:, :17] = -1
    rag = build_rag(T(L, cuda), R, T(sc["image"], cuda))
    k, b, area, per = oc.build_rag(L, R)
    assert np.array_equal(keys_np(rag.edge_keys), k) and np.array_equal(rag.boundary_len.cpu().numpy().view(np.uint32), b)
    assert np.array_equal(rag.area.cpu().numpy(), area) and np.array_equal(rag.perimeter.cpu().numpy(), per)
    s, q = oc.pool_bands(L, sc["image"], R)
    assert np.array_equal(rag.band_sum.cpu().numpy().view(np.uint64), s)
    assert np.array_equal(rag.band_sumsq.cpu().numpy().view(np.uint64), q)
    res = merge_scene(T(sc["labels"], cuda), T(sc["feats"], cuda), 0.5, n_regions=R, image=T(sc["image"], cuda),
                      xs=T(sc["xs"], cuda), ys=T(sc["ys"], cuda))
    root = res.root.cpu().numpy()
    assert np.array_equal(res.labels.cpu().numpy(), oc.relabel(sc["labels"], root))
    k2, b2, area2, per2 = oc.build_rag(res.labels.cpu().numpy(), R)
    roots = np.unique(root)
    assert np.array_equal(keys_np(res.edge_keys), k2) and np.array_equal(res.boundary_len.cpu().numpy().view(np.uint32), b2)
    assert np.array_equal(res.area.cpu().numpy()[roots], area2[roots])
    assert np.array_equal(res.perimeter.cpu().numpy()[roots], per2[roots])
    # the selected edges of the first round, recomputed on the CPU from the GPU's own scores, give the same roots
    g0 = merge_scene(T(sc["labels"], cuda), T(sc["feats"], cuda), 0.5, n_regions=R, xs=T(sc["xs"], cuda), ys=T(sc["ys"], cuda),
                     max_rounds=0)
    sel = g0.scores.cpu().numpy() < 0.5
    kk = keys_np(g0.edge_keys)[sel]
    r1 = oc.min_roots(R, (kk >> np.uint64(32)).astype(np.int32), (kk & np.uint64(0xFFFFFFFF)).astype(np.int32))
    if res.rounds == 1:
        assert np.array_equal(r1, root)


@pytest.mark.parametrize("D", [7, 100, 128])
def test_pool_points_with_means_in_one_pass(cuda, D):
    """dm_pool_points_csr_mean = dm_pool_points_csr + dm_region_mean, bit for bit (sum, cnt, mean, norm2), including
    regions without points (NaN mean and norm)."""
    import torch
    from deepmerge_b200 import raster as rs
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(D)
    R, N = 5000, 17000
    rop = rng.integers(0, R - 40, N).astype(np.int32)              # the last 40 regions stay empty
    feats = rng.standard_normal((N, D)).astype(np.float32)
    d_rop, d_f = T(rop, cuda), T(feats, cuda)
    off, ids = rs.csr_from_region_of_point(d_rop, R)
    s1, c1 = rs.pool_points_csr(off, ids, d_f)
    m1, n1 = rs.region_mean(s1, c1)
    s2 = torch.empty_like(s1); c2 = torch.empty_like(c1); m2 = torch.empty_like(m1); n2 = torch.empty_like(n1)
    st = torch.cuda.current_stream().cuda_stream
    L.check(L.dm_pool_points_csr_mean(off.data_ptr(), ids.data_ptr(), d_f.data_ptr(), D, R, D, s2.data_ptr(), c2.data_ptr(),
                                      m2.data_ptr(), n2.data_ptr(), st), "dm_pool_points_csr_mean")
    torch.cuda.synchronize()
    assert torch.equal(s1, s2) and torch.equal(c1, c2)
    assert np.array_equal(m1.cpu().numpy(), m2.cpu().numpy(), equal_nan=True)
    assert np.array_equal(n1.cpu().numpy(), n2.cpu().numpy(), equal_nan=True)
    assert np.isnan(m2[-40:].cpu().numpy()).all()
    assert L.dm_pool_points_csr_mean(off.data_ptr(), ids.data_ptr(), d_f.data_ptr(), 200, R, 200, s2.data_ptr(), c2.data_ptr(),
                                     m2.data_ptr(), n2.data_ptr(), st) == -4          # DM_ERR_UNSUPPORTED: D > 128
