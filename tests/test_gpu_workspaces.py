"""GPU: every entry point that takes a workspace stays inside the bytes its query reports.  Each call gets as its
workspace the first `query` bytes of a longer buffer filled with a sentinel; it must return DM_OK, leave every byte from
`query` on holding the sentinel, and give what the package's wrapper gives -- or, for an entry point without one, what
the same call gives on a workspace of exactly `query` bytes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

SENTINEL = 0xA7
PAD = 1 << 20
# capacities below one sort tile and above many, neither a multiple of 256 nor of the 2048-pair sort tile
SIZES = [257, 97969]


@pytest.fixture(scope="module")
def L(cuda):
    from deepmerge_b200._lib import lib
    return lib()


def p(t):
    return None if t is None else t.data_ptr()


def in_queried_ws(query, call):
    """call(ws, ws_bytes) with ws the first `query` bytes of a sentinel-filled buffer PAD bytes longer"""
    buf = torch.full((query + PAD,), SENTINEL, dtype=torch.uint8, device="cuda")
    assert call(p(buf), query) == 0
    torch.cuda.synchronize()
    written = (buf[query:] != SENTINEL).nonzero()
    assert written.numel() == 0, "byte %d written, the query reports %d" % (query + int(written[0]), query)


def in_exact_ws(query, call):
    ws = torch.empty(query, dtype=torch.uint8, device="cuda")
    assert call(p(ws), query) == 0
    torch.cuda.synchronize()


def merge_state(R, seed):
    """A compressed union-find forest over R regions (every component's root is its minimum id)."""
    rng = np.random.default_rng(seed)
    comp = rng.integers(0, R // 3 + 1, R)
    first = np.full(comp.max() + 1, R)
    np.minimum.at(first, comp, np.arange(R))
    return torch.from_numpy(first[comp].astype(np.int32)).cuda(), rng


def assert_same(a, b):
    """bit for bit"""
    assert a.shape == b.shape and a.dtype == b.dtype
    assert torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


@pytest.mark.parametrize("H,W,R", [(64, 80, 40), (1000, 1000, 20000)])
def test_rag_build(L, H, W, R):
    from deepmerge_b200 import build_rag
    from deepmerge_b200.synth import synth_scene
    sc = synth_scene(H, W, R, C=3, device="cuda")
    R, C, cap = sc.n_regions, 3, 2 * H * W + 1          # room for every boundary pixel pair: no overflow
    want = build_rag(sc.labels, R, sc.image, capacity=cap)
    z = lambda *s: torch.zeros(*s, dtype=torch.int64, device="cuda")
    area, border, bsum, bsq, counts = z(R), z(R), z((R, C)), z((R, C)), z(4)
    keys = torch.empty(cap, dtype=torch.int64, device="cuda")
    blen = torch.empty(cap, dtype=torch.int32, device="cuda")
    in_queried_ws(L.dm_rag_workspace_bytes(cap), lambda ws, n: L.dm_rag_build(
        p(sc.labels), H, H, W, W, p(sc.image), C, W * C, R, 1, 1, p(area), p(border), p(bsum), p(bsq), p(keys), p(blen),
        cap, p(counts), ws, n, None))
    E = int(counts[0])
    assert counts[2:].tolist() == [0, 0] and E == want.n_edges
    for got, w in ((keys[:E], want.edge_keys), (blen[:E], want.boundary_len), (area, want.area), (border, want.border),
                   (bsum, want.band_sum), (bsq, want.band_sumsq)):
        assert_same(got, w)


@pytest.mark.parametrize("n", SIZES)
def test_edges_sort_unique(L, n):
    from deepmerge_b200 import merge_edge_lists
    rng = np.random.default_rng(n)
    R = n // 3 + 2
    lo, hi = rng.integers(0, R, n), rng.integers(0, R, n)
    keys = torch.from_numpy(((np.minimum(lo, hi) << 32) | np.maximum(lo, hi)).astype(np.int64)).cuda()
    lens = torch.from_numpy(rng.integers(1, 1000, n).astype(np.int32)).cuda()
    want_k, want_l = merge_edge_lists(keys, lens, R)
    k, l = keys.clone(), lens.clone()
    cnt = torch.tensor([n, -1], dtype=torch.int64, device="cuda")
    in_queried_ws(L.dm_edges_unique_workspace_bytes(n), lambda ws, wsb: L.dm_edges_sort_unique(
        p(k), p(l), p(cnt), n, R, p(cnt[1:]), ws, wsb, None))
    E = int(cnt[1])
    assert_same(k[:E], want_k)
    assert_same(l[:E], want_l)


@pytest.mark.parametrize("n", SIZES)
def test_csr_build(L, n):
    from deepmerge_b200 import csr_from_region_of_point
    R = n // 5 + 3
    rop = torch.from_numpy(np.random.default_rng(n).integers(-1, R, n).astype(np.int32)).cuda()
    want_off, want_ids = csr_from_region_of_point(rop, R)
    off = torch.empty(R + 1, dtype=torch.int64, device="cuda")
    ids = torch.empty(n, dtype=torch.int32, device="cuda")
    in_queried_ws(L.dm_csr_workspace_bytes(n, R), lambda ws, wsb: L.dm_csr_build(p(rop), n, R, p(off), p(ids), ws, wsb,
                                                                                 None))
    assert_same(off, want_off)
    m = int(off[R])
    assert_same(ids[:m], want_ids[:m])


@pytest.mark.parametrize("masked", [False, True], ids=["all", "mask"])
@pytest.mark.parametrize("R", SIZES)
def test_merge_apply_masked(L, R, masked):
    D = 5
    parent, rng = merge_state(R, R)
    mask = torch.from_numpy(rng.integers(0, 2, R).astype(np.uint8)).cuda() if masked else None
    state = [torch.ones(R, dtype=torch.uint8, device="cuda"), torch.zeros(R, dtype=torch.uint8, device="cuda"),
             torch.from_numpy(rng.standard_normal((R, D)).astype(np.float32)).cuda(),
             torch.from_numpy(rng.integers(1, 50, R).astype(np.int32)).cuda(),
             torch.from_numpy(rng.integers(1, 500, R)).cuda(), torch.from_numpy(rng.integers(4, 100, R)).cuda(),
             torch.full((1,), -1, dtype=torch.int64, device="cuda")]
    runs = []
    for run in (in_exact_ws, in_queried_ws):
        s = [t.clone() for t in state]
        alive, changed, sum_, cnt, area, perim, n_merged = (p(t) for t in s)
        run(L.dm_merge_apply_workspace_bytes(R), lambda ws, wsb: L.dm_merge_apply_masked(
            p(parent), alive, changed, sum_, cnt, area, perim, R, D, n_merged, p(mask), ws, wsb, None))
        runs.append(s)
    assert int(runs[1][6]) > 0
    for a, b in zip(*runs):
        assert_same(a, b)


@pytest.mark.parametrize("with_scores", [False, True], ids=["lens", "scores"])
@pytest.mark.parametrize("cap", SIZES)
def test_edges_rekey(L, cap, with_scores):
    R = cap // 2 + 5
    parent, rng = merge_state(R, cap + 1)
    lo, hi = rng.integers(0, R, 2 * cap), rng.integers(0, R, 2 * cap)
    keys = np.unique(((np.minimum(lo, hi) << 32) | np.maximum(lo, hi))[lo != hi])[:cap - 3]   # a device count < cap
    E = keys.size
    state = [torch.zeros(cap, dtype=torch.int64, device="cuda"), torch.zeros(cap, dtype=torch.int32, device="cuda"),
             torch.zeros(cap, dtype=torch.float32, device="cuda"), torch.tensor([E], dtype=torch.int64, device="cuda"),
             torch.from_numpy(rng.integers(10**6, 10**7, R)).cuda()]
    state[0][:E] = torch.from_numpy(keys.astype(np.int64)).cuda()
    state[1][:E] = torch.from_numpy(rng.integers(1, 100, E).astype(np.int32)).cuda()
    state[2][:E] = torch.from_numpy(rng.standard_normal(E).astype(np.float32)).cuda()
    runs = []
    for run in (in_exact_ws, in_queried_ws):
        s = [t.clone() for t in state]
        keys_t, lens, scores, n_dev, perim = s
        run(L.dm_edges_rekey_workspace_bytes(cap), lambda ws, wsb: L.dm_edges_rekey(
            p(parent), p(keys_t), p(lens), p(scores) if with_scores else None, p(n_dev), cap, R, p(perim), ws, wsb, None))
        runs.append(s)
    m = int(runs[1][3])
    assert 0 < m < E
    for a, b in zip(*runs):
        assert_same(a[:m] if a.numel() == cap else a, b[:m] if b.numel() == cap else b)


@pytest.mark.parametrize("R", SIZES)
def test_compact_roots(L, R):
    from deepmerge_b200 import compact_roots
    root, _ = merge_state(R, R + 2)
    want, want_n = compact_roots(root)
    out = torch.empty(R, dtype=torch.int32, device="cuda")
    n = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    in_queried_ws(L.dm_compact_roots_workspace_bytes(R), lambda ws, wsb: L.dm_compact_roots(p(root), R, p(out), p(n), ws,
                                                                                            wsb, None))
    assert int(n) == want_n
    assert_same(out, want)


@pytest.mark.parametrize("cap", SIZES)
def test_sort_edges(L, cap):
    rng = np.random.default_rng(cap + 3)
    R = cap // 4 + 7
    n = cap - 2
    lo, hi = rng.integers(0, R, n), rng.integers(0, R, n)
    state = [torch.zeros(cap, dtype=torch.int64, device="cuda"),
             torch.from_numpy(np.arange(cap, dtype=np.int32)).cuda(), torch.tensor([n], dtype=torch.int64, device="cuda")]
    state[0][:n] = torch.from_numpy(((lo << 32) | hi).astype(np.int64)).cuda()
    runs = []
    for run in (in_exact_ws, in_queried_ws):
        k, v, nd = [t.clone() for t in state]
        run(L.dm_sort_edges_workspace_bytes(cap), lambda ws, wsb: L.dm_sort_edges(p(k), p(v), p(nd), cap, R, ws, wsb, None))
        runs.append((k[:n], v[:n]))
    assert bool((runs[1][0][1:] >= runs[1][0][:-1]).all())
    for a, b in zip(*runs):
        assert_same(a, b)


@pytest.mark.parametrize("cap", SIZES)
def test_scan_exclusive_u32(L, cap):
    n = cap - 1
    x = torch.from_numpy(np.random.default_rng(cap).integers(0, 5, cap).astype(np.int32)).cuda()
    nd = torch.tensor([n], dtype=torch.int64, device="cuda")
    runs = []
    for run in (in_exact_ws, in_queried_ws):
        out = torch.full((cap,), -1, dtype=torch.int32, device="cuda")
        tot = torch.full((1,), -1, dtype=torch.int64, device="cuda")
        run(L.dm_scan_workspace_bytes(cap), lambda ws, wsb: L.dm_scan_exclusive_u32(p(x), p(out), p(nd), cap, p(tot), ws,
                                                                                    wsb, None))
        runs.append((out, tot))
    assert int(runs[1][1]) == int(x[:n].sum())
    for a, b in zip(*runs):
        assert_same(a, b)


@pytest.mark.parametrize("H,W,R", [(37, 61, 9), (300, 257, 400)])
def test_polygonize(L, H, W, R):
    from deepmerge_b200 import polygonize
    from deepmerge_b200.polygons import default_capacity
    from deepmerge_b200.synth import synth_scene
    sc = synth_scene(H, W, R, C=0, device="cuda", with_image=False)
    R, cap = sc.n_regions, default_capacity(sc.n_regions, H, W)
    want = polygonize(sc.labels, R, capacity=cap)
    ring_cap = cap // 4
    e = lambda *s, dt: torch.empty(*s, dtype=dt, device="cuda")
    bufs = [e(ring_cap, dt=torch.int32), e(ring_cap + 1, dt=torch.int64), e(ring_cap, dt=torch.int64),
            e((cap, 2), dt=torch.int32), e(R + 1, dt=torch.int64)]
    counts = torch.zeros(4, dtype=torch.int64, device="cuda")
    in_queried_ws(L.dm_polygonize_workspace_bytes(H, W, R, cap), lambda ws, wsb: L.dm_polygonize(
        p(sc.labels), H, W, W, R, cap, *[p(b) for b in bufs], p(counts), ws, wsb, None))
    k, v = int(counts[0]), int(counts[1])
    assert counts[3] == 0 and int(counts[2]) == want.boundary_sides
    for got, w in ((bufs[0][:k], want.ring_region), (bufs[1][:k + 1], want.ring_offsets), (bufs[2][:k], want.ring_area),
                   (bufs[3][:v], want.vertices), (bufs[4], want.region_rings)):
        assert_same(got, w)
