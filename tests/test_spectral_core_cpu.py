"""CPU: merge by spectral and shape heterogeneity.

deepmerge_b200/csrc/spectral_core.cuh holds the per-edge fusion arithmetic the score kernel of dm_score_spectral calls;
the same header is compiled here with g++ (tests/spectral_core_host.cpp runs the kernel's loop sequentially) and
checked bit for bit against spectral_fusion of tests/spectral_oracle.py on random statistics and extremes.  The
oracle's merge loop (merge_spectral) is checked against itself: its fixed point, its incremental statistics against a
fresh pass over the relabelled raster, and a hand-computed graph."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_np as o

import spectral_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("spectral_core") / "libspectral_core_host.so")
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC", "-o", so,
                        os.path.join(HERE, "spectral_core_host.cpp")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(so)
    lib.score_spectral_host.restype = ctypes.c_int
    lib.score_spectral_host.argtypes = [ctypes.c_void_p] * 2 + [ctypes.c_long] + [ctypes.c_void_p] * 4 + [ctypes.c_int] + \
        [ctypes.c_void_p] * 2 + [ctypes.c_float] * 2 + [ctypes.c_void_p]

    def run(g, w_shape, w_cmpct, band_w=None):
        a = {k: np.ascontiguousarray(v) for k, v in g.items()}
        bw = None if band_w is None else np.ascontiguousarray(band_w, np.float32)
        out = np.full(a["keys"].shape[0], np.nan, np.float32)
        lib.score_spectral_host(a["keys"].ctypes.data, a["blen"].ctypes.data, a["keys"].shape[0], a["area"].ctypes.data,
                                a["perim"].ctypes.data, a["bsum"].ctypes.data, a["bsq"].ctypes.data, a["bsum"].shape[1],
                                a["bbox"].ctypes.data, None if bw is None else bw.ctypes.data, w_shape, w_cmpct,
                                out.ctypes.data)
        return out
    return run


def random_stats(rng, R, C, E, n_max=10 ** 6, extremes=True):
    """Plausible integer statistics of R regions and E edges: band sums with S^2 / n <= Q <= 255 S, perimeters and
    boundary lengths with L <= min(l_a, l_b), boxes of at least n pixels.  With extremes: 1-pixel regions, bands
    saturated at 0 and 255, regions of up to 10^8 pixels."""
    n = rng.integers(1, n_max + 1, R).astype(np.int64)
    if extremes:
        n[: R // 8] = 1
        n[R // 8: R // 6] = rng.integers(10 ** 7, 10 ** 8 + 1, R // 6 - R // 8)
        n[R // 6] = 10 ** 8
    S = np.empty((R, C), np.int64)
    Q = np.empty((R, C), np.int64)
    for c in range(C):
        s = (rng.random(R) * (255 * n + 1)).astype(np.int64)
        s = np.minimum(s, 255 * n)
        lo_q = np.array([-(-int(v) * int(v) // int(m)) for v, m in zip(s, n)], np.int64)     # ceil(S^2 / n), exact
        q = lo_q + (rng.random(R) * (255 * s - lo_q + 1)).astype(np.int64)
        S[:, c], Q[:, c] = s, np.minimum(q, 255 * s)
    if extremes:
        S[: R // 16], Q[: R // 16] = 0, 0                           # black
        S[R // 16: R // 8] = 255 * n[R // 16: R // 8, None]         # saturated white 1-pixel regions
        Q[R // 16: R // 8] = 255 * 255 * n[R // 16: R // 8, None]
    side = np.ceil(np.sqrt(n)).astype(np.int64)
    w = side + rng.integers(0, 5, R)
    h = np.maximum(-(-n // w), 1) + rng.integers(0, 5, R)
    x0, y0 = rng.integers(0, 1000, R), rng.integers(0, 1000, R)
    bbox = np.stack([x0, y0, x0 + w - 1, y0 + h - 1], 1).astype(np.int32)
    perim = (4 * side + rng.integers(0, 40, R) * (n > 1)).astype(np.int64)
    a = rng.integers(0, R - 1, E)
    b = a + 1 + (rng.random(E) * (R - 1 - a)).astype(np.int64)
    keys = o.pack_keys(a, b)
    L = np.maximum(1, (rng.random(E) * np.minimum(perim[a], perim[b])).astype(np.int64)).astype(np.uint32)
    return dict(keys=keys, blen=L, area=n, perim=perim, bsum=S.astype(np.uint64), bsq=Q.astype(np.uint64), bbox=bbox)


def oracle(g, w_shape, w_cmpct, band_w=None):
    return so.spectral_fusion(g["area"], g["perim"], g["bsum"], g["bsq"], g["bbox"], g["keys"], g["blen"], w_shape, w_cmpct,
                             band_w)


def bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


@pytest.mark.parametrize("C", range(1, 9))
def test_core_matches_the_oracle_bit_for_bit(host, C):
    rng = np.random.default_rng(100 + C)
    g = random_stats(rng, 400, C, 3000)
    bw = rng.random(C).astype(np.float32) * 2
    for w_shape in (0.0, 0.1, 0.9, 1.0):
        for w_cmpct in (0.0, 0.5, 1.0):
            for band_w in (None, bw):
                want = oracle(g, w_shape, w_cmpct, band_w)
                assert np.isfinite(want).all()
                assert np.array_equal(bits(host(g, w_shape, w_cmpct, band_w)), bits(want)), (w_shape, w_cmpct)


def test_core_small_regions_and_negative_shape_terms(host):
    """Two 10 x 5 halves of a 10 x 10 square: merging them lowers the shape heterogeneity (h_cmpct < 0, h_smooth = 0),
    so with w_shape = 1 the fusion value is negative; 1-pixel regions of identical colour fuse at exactly 0."""
    g = dict(keys=o.pack_keys([0, 2], [1, 3]), blen=np.array([10, 1], np.uint32), area=np.array([50, 50, 1, 1], np.int64),
             perim=np.array([30, 30, 4, 4], np.int64), bsum=np.array([[500], [500], [7], [7]], np.uint64),
             bsq=np.array([[5000], [5000], [49], [49]], np.uint64),
             bbox=np.array([[0, 0, 9, 4], [0, 5, 9, 9], [20, 0, 20, 0], [21, 0, 21, 0]], np.int32))
    for w_cmpct in (0.0, 0.5, 1.0):
        want = oracle(g, 1.0, w_cmpct)
        assert np.array_equal(bits(host(g, 1.0, w_cmpct)), bits(want))
        h_cmpct = 100 * 40 / 10 - 2 * (50 * 30 / np.sqrt(50))
        assert want[0] == np.float32(w_cmpct * h_cmpct) and (w_cmpct == 0 or want[0] < 0)
    assert oracle(g, 0.0, 0.5)[1] == 0 and oracle(g, 0.0, 0.5)[0] == 0


def test_core_random_shapes_are_often_negative(host):
    rng = np.random.default_rng(7)
    g = random_stats(rng, 300, 3, 2000, n_max=400, extremes=False)
    want = oracle(g, 1.0, 0.5)
    assert (want < 0).sum() > 10
    assert np.array_equal(bits(host(g, 1.0, 0.5)), bits(want))


# ------------------------------------------------------------------------------------------
# the oracle's merge loop
# ------------------------------------------------------------------------------------------
def strips(values, width=4, height=4):
    """One row of vertical strips, strip i of uniform colour values[i] (C = 1)."""
    lab = np.repeat(np.arange(len(values), dtype=np.int32), width)[None, :].repeat(height, 0)
    img = np.asarray(values, np.uint8)[lab][..., None]
    return lab, img


def test_hand_built_chain_gives_the_hand_computed_rounds():
    """Four uniform 4 x 4 strips of colour 0, 1, 3, 7 and w_shape = 0: two uniform regions fuse at |v_a - v_b| sqrt(n_a n_b),
    so the edges start at 16, 32, 64.  Round 1 merges (0, 1) only: the best edge of region 2 is (1, 2), not (2, 3).
    Round 2: {0, 1} + 2 fuses at 48 sqrt(14) / 3 - 32 / 2 = 43.87 < 64, merged.  Round 3: the whole row fuses at
    64 sqrt(115) / 4 - 48 sqrt(14) / 3 = 111.7: merged under scale 12 (threshold 144), not under scale 10 (100)."""
    lab, img = strips([0, 1, 3, 7])
    g = so.merge_scene_spectral(lab, img, 4, 10.0, w_shape=0.0, max_rounds=0)
    assert np.array_equal(g["scores"], np.float32([16, 32, 64]))
    g = so.merge_scene_spectral(lab, img, 4, 10.0, w_shape=0.0)
    assert g["rounds"] == 2 and g["merges"] == 2 and g["root"].tolist() == [0, 0, 0, 3]
    assert np.isclose(g["scores"][0], 64 * np.sqrt(115) / 4 - 48 * np.sqrt(14) / 3, rtol=1e-6)
    g = so.merge_scene_spectral(lab, img, 4, 12.0, w_shape=0.0)
    assert g["rounds"] == 3 and g["merges"] == 3 and g["root"].tolist() == [0, 0, 0, 0] and g["keys"].size == 0
    g = so.merge_scene_spectral(lab, img, 4, 12.0, w_shape=0.0, max_rounds=1)
    assert g["rounds"] == 1 and g["root"].tolist() == [0, 0, 2, 3]


def test_equal_scores_resolve_by_edge_index():
    lab, img = strips([0, 1, 0])                                     # both edges fuse at 16
    g = so.merge_scene_spectral(lab, img, 3, 4.5, w_shape=0.0, max_rounds=1)
    assert g["root"].tolist() == [0, 0, 2]
    keys = o.pack_keys([0, 0, 1, 2], [1, 2, 2, 3])                  # a triangle and a tail, every score equal
    assert so.select_mutual(np.float32([1, 1, 1, 1]), keys, 2.0, 4).tolist() == [True, False, False, False]
    assert so.select_mutual(np.float32([1, 1, 0.5, 1]), keys, 2.0, 4).tolist() == [False, False, True, False]
    assert so.select_mutual(np.float32([0.0, -0.0, 1, 1]), keys, 2.0, 4).tolist() == [True, False, False, False]
    assert so.select_mutual(np.float32([np.nan, 1, 1, 2]), keys, 2.0, 4).tolist() == [False, True, False, False]
    assert not so.select_mutual(np.float32([2, 2, 2, 2]), keys, 2.0, 4).any()      # threshold is exclusive


@pytest.mark.parametrize("C,shape,nodata", [(1, 0.1, False), (3, 0.5, True), (4, 0.0, False)])
def test_oracle_fixed_point_and_incremental_statistics(C, shape, nodata):
    sc = o.synth_scene(96, 128, 150, C=C, seed=11 + C)
    lab, img, R = sc["labels"].copy(), sc["image"], sc["n_regions"]
    if nodata:
        lab[20:40, 30:70] = -1
        lab[:, :3] = -1
    scale = 25.0
    g = so.merge_scene_spectral(lab, img, R, scale, w_shape=shape)
    assert g["rounds"] > 1 and g["merges"] > 0
    thr = np.float32(scale * scale)
    # fixed point: with f recomputed from the final statistics no adjacent pair fuses below scale^2
    f = so.spectral_fusion(g["area"], g["perim"], g["bsum"], g["bsq"], g["bbox"], g["keys"], g["blen"], shape, 0.5)
    assert np.array_equal(f, g["scores"]) and not (f < thr).any()
    # the incremental statistics equal a fresh pass over the relabelled raster, at every root
    keys, blen, area, perim = o.build_rag(g["labels"], R)
    s, q = o.pool_bands(g["labels"], img, R)
    box = o.region_bbox(g["labels"], R)
    roots = np.nonzero(g["root"] == np.arange(R))[0]
    roots = roots[area[roots] > 0]
    assert np.array_equal(keys, g["keys"]) and np.array_equal(blen, g["blen"])
    assert np.array_equal(area[roots], g["area"][roots]) and np.array_equal(perim[roots], g["perim"][roots])
    assert np.array_equal(s[roots], g["bsum"][roots]) and np.array_equal(q[roots], g["bsq"][roots])
    assert np.array_equal(box[roots], g["bbox"][roots])
    assert g["merges"] == R - len(np.unique(g["root"]))
