"""Region statistics compared bit for bit: point pooling (dm_pool_points_csr / _tile / _mean), region means and norms
(dm_region_mean), merged sums and counts (dm_merge_apply / _masked), union-find (dm_uf_union / dm_uf_compress), edge
selection (dm_merge_select_l2 / _mlp) and the re-keyed edge list with its carried scores (dm_edges_rekey), each against
a restatement of the order the header promises (include/deepmerge_b200.h: sequential fp32 accumulation in membership
order, members added in ascending id, norms as per-lane FMA chains and an xor butterfly).

Inputs are standard-normal fp32, not integers: the order of summation is what is under test.  A reordered sum, a
skipped chunk of point ids, a mul+add in place of an FMA or a merged sum that starts from zero changes result bits, and
the CPU tests below show that each restatement tells such variants apart on inputs like these.

Each GPU case asserts the path its inputs take, restating the grid rule grid_for of csrc/common.cuh and the path
rules of csrc/pool.cu and csrc/prims.cu; the test ids name the path.
"""
import threading
from fractions import Fraction

import numpy as np
import pytest

from oracle import oracle_np as o
from test_gpu_scorers_exact import SENTINEL, T, num_sms, same
from test_gpu_sharded import FakeDist

INT64_MAX = np.iinfo(np.int64).max
SENT_U32 = 0xDEADBEEF                               # bits of SENTINEL
SENT_I32 = int(np.array([SENT_U32], np.uint32).view(np.int32)[0])
HUB_MIN, HUB_MAX, HUB_CAP = 48, 4096, 1024          # edge_unique_hashed (csrc/prims.cu)
HUB_MAX_SORT = 2048                                 # bucket_sort_fused (csrc/prims.cu)


# ------------------------------------------------------------------------------------------
# restatements
# ------------------------------------------------------------------------------------------
def grid_for(items, S, threads=256, per_sm=8):
    """csrc/common.cuh: one thread per item, at most per_sm blocks per SM."""
    return max(1, min(-(-items // threads), S * per_sm))


def warps_for(R, S):
    """Warps of a one-warp-per-item kernel launched with grid_for(R * 32) blocks of 256 threads."""
    return grid_for(R * 32, S) * 8


def fma32(a, b, c):
    """fp32 a * b + c rounded once (__fmaf_rn).  The float64 product of two fp32 values is exact; TwoSum of it with c
    gives the float64 sum s and its rounding error, and float32(s) is the correctly rounded result unless s is an fp32
    midpoint with a nonzero error, where the error's sign picks the side."""
    a = np.asarray(a, np.float32).astype(np.float64)
    b = np.asarray(b, np.float32).astype(np.float64)
    c = np.asarray(c, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        p = a * b
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)
        r = s.astype(np.float32)
        lo = np.where(r.astype(np.float64) > s, np.nextafter(r, np.float32(-np.inf)), r)
        hi = np.nextafter(lo, np.float32(np.inf))
        mid = (lo.astype(np.float64) + hi.astype(np.float64)) / 2          # exact in float64
        tie = (s == mid) & (err != 0)
        r = np.where(tie & (err > 0), hi, np.where(tie & (err < 0), lo, r))
    return r.astype(np.float32)


def muladd32(a, b, c):
    """The contraction the kernels must NOT use: fp32 product, then fp32 sum (two roundings)."""
    return np.asarray(a, np.float32) * np.asarray(b, np.float32) + np.asarray(c, np.float32)


def norm2_ref(mean, fma=fma32, reverse=False):
    """norm2 as region_mean_kernel / pool_points_kernel form it: lane l chains fma(v, v, acc) over d = l + 32 k in
    ascending k, then the xor butterfly 16, 8, 4, 2, 1 (fp32 adds) and lane 0's value."""
    mean = np.asarray(mean, np.float32)
    R, D = mean.shape
    lanes = np.zeros((R, 32), np.float32)
    ks = list(range(-(-D // 32)))
    for k in (ks[::-1] if reverse else ks):
        w = min(32, D - 32 * k)
        v = mean[:, 32 * k:32 * k + w]
        lanes[:, :w] = fma(v, v, lanes[:, :w])
    with np.errstate(invalid="ignore"):
        for off in (16, 8, 4, 2, 1):
            lanes = lanes + lanes[:, np.arange(32) ^ off]
    return lanes[:, 0]


def pool_ref(offsets, ids, feats):
    """(sum, cnt, mean, norm2): oracle_np's sequential fp32 pooling in the given membership order."""
    s, c, _ = o.pool_points_csr(offsets, ids, feats)
    m = o.region_mean(s, c)
    return s, c, m, norm2_ref(m)


def merge_apply_ref(parent, alive, sum_, cnt, area, perim, root_mask=None, descending=False):
    """dm_merge_apply(_masked): every alive region x with parent[x] != x is absorbed -- cnt / area / perimeter added to
    its root for every root; the root's sum (roots with root_mask set, all without a mask) starts from its own row and
    adds the members' rows one fp32 addition at a time in ascending member id (descending=True: the order it must not
    use)."""
    R = parent.shape[0]
    sum_, cnt, area, perim, alive = sum_.copy(), cnt.copy(), area.copy(), perim.copy(), alive.copy()
    moved = np.nonzero((alive != 0) & (parent != np.arange(R)))[0]
    tg = parent[moved]
    changed = np.zeros(R, np.uint8)
    changed[tg] = 1
    np.add.at(cnt, tg, cnt[moved])
    np.add.at(area, tg, area[moved])
    np.add.at(perim, tg, perim[moved])
    alive[moved] = 0
    listed = moved if root_mask is None else moved[root_mask[tg] != 0]
    if descending:
        listed = listed[::-1]
    mv = listed[np.argsort(parent[listed], kind="stable")]
    root = parent[mv]
    starts = np.r_[0, np.nonzero(np.diff(root))[0] + 1] if mv.size else np.zeros(0, np.int64)
    lens = np.diff(np.r_[starts, mv.size])
    for k in range(int(lens.max(initial=0))):
        s = starts[lens > k] + k
        sum_[root[s]] = sum_[root[s]] + sum_[mv[s]]
    return dict(sum=sum_, cnt=cnt, area=area, perim=perim, alive=alive, changed=changed, n_merged=moved.size)


def components(rng, R, sizes):
    """parent of min-root components of the given sizes over randomly scattered ids; the other ids stay singletons."""
    perm = rng.permutation(R)
    parent = np.arange(R, dtype=np.int64)
    pos = 0
    for s in sizes:
        m = perm[pos:pos + s]
        pos += s
        parent[m] = m.min()
    assert pos <= R
    return parent


def csr_inputs(rng, R, pts, specials, D, ld, shuffled):
    """Region r gets 0..5 points, the `specials` get `pts`.  Feature rows are standard normal, columns D..ld-1 of the
    wider array are NaN (a read past D shows), 50 rows belong to no region; shuffled: ids in random, not ascending,
    order."""
    cnt = rng.integers(0, 6, R)
    cnt[specials] = pts
    N = int(cnt.sum())
    rows = N + 50
    wide = rng.standard_normal((rows, ld)).astype(np.float32)
    wide[:, D:] = np.nan
    ids = (rng.permutation(rows)[:N] if shuffled else np.arange(N)).astype(np.int32)
    offsets = np.zeros(R + 1, np.int64)
    np.cumsum(cnt, out=offsets[1:])
    return offsets, ids, wide


# ------------------------------------------------------------------------------------------
# CPU: the restatements are exact, and the exact comparisons have teeth
# ------------------------------------------------------------------------------------------
def fma_fraction(a, b, c):
    v = Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))
    f = np.float32(float(v))
    cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
    return min(cands, key=lambda x: (abs(Fraction(float(x)) - v), int(np.array(x, np.float32).view(np.uint32)) & 1))


def test_fma32_is_correctly_rounded():
    """fma32 against exact rational arithmetic on random triples and on triples built to sit a hair from an fp32
    midpoint: c has an odd last bit and a * b = ulp(c) / 2 (1 - 2^-46), so the float64 sum is the midpoint itself and
    rounding it once more (ties to even) lands on the wrong side, in both directions of the sign."""
    rng = np.random.default_rng(0)
    n, m = 3000, 1000
    mant = (2 ** 23 + 2 * rng.integers(0, 2 ** 22, m) + 1).astype(np.float64)       # odd 24-bit significands
    e = rng.integers(-40, 40, m)
    sign = np.where(np.arange(m) % 2 == 0, 1.0, -1.0)
    c_hard = (sign * mant * np.exp2(e - 23)).astype(np.float32)
    a_hard = (sign * (1 + 2.0 ** -23)).astype(np.float32)
    b_hard = ((1 - 2.0 ** -23) * np.exp2(e - 24)).astype(np.float32)          # ulp(c) / 2 (1 - 2^-23)
    a = np.r_[rng.standard_normal(n), a_hard].astype(np.float32)
    b = np.r_[rng.standard_normal(n), b_hard].astype(np.float32)
    c = np.r_[rng.standard_normal(n) * np.exp2(rng.integers(-30, 30, n)), c_hard].astype(np.float32)
    got = fma32(a, b, c)
    double_rounded = (a.astype(np.float64) * b + c).astype(np.float32)
    assert (got[n:] != double_rounded[n:]).all()                    # the midpoint correction decides every hard case
    for i in range(n + m):
        assert got[i].view(np.uint32) == fma_fraction(a[i], b[i], c[i]).view(np.uint32), i


def test_norm2_ref_is_discriminating():
    rng = np.random.default_rng(1)
    mean = rng.standard_normal((2000, 100)).astype(np.float32)
    want = norm2_ref(mean)
    differ = lambda x: float(np.mean(x.view(np.uint32) != want.view(np.uint32)))
    assert differ(norm2_ref(mean, fma=muladd32)) > 0.05
    assert differ(np.sum(mean.astype(np.float64) ** 2, 1).astype(np.float32)) > 0.1
    assert differ(norm2_ref(mean, reverse=True)) > 0.05
    ints = rng.integers(-8, 9, (500, 260)).astype(np.float32)       # exact arithmetic: every order agrees
    assert np.array_equal(norm2_ref(ints), (ints.astype(np.float64) ** 2).sum(1).astype(np.float32))
    nan = mean[:3].copy()
    nan[1] = np.nan
    assert np.isnan(norm2_ref(nan)[1]) and np.isfinite(norm2_ref(nan)[[0, 2]]).all()


def test_pool_ref_is_discriminating():
    rng = np.random.default_rng(2)
    feats = rng.standard_normal((300, 65)).astype(np.float32)
    ids = rng.permutation(300)[:100].astype(np.int32)               # one region of 100 points, 4 chunks of ids
    off = np.array([0, 100], np.int64)
    s = o.pool_points_csr(off, ids, feats)[0][0]
    acc = np.zeros(65, np.float32)
    for i in ids:                                                   # the left fold, one fp32 row addition at a time
        acc = acc + feats[i]
    assert np.array_equal(s.view(np.uint32), acc.view(np.uint32))
    assert not np.array_equal(s, o.pool_points_csr(off, ids[::-1].copy(), feats)[0][0])
    first32 = o.pool_points_csr(np.array([0, 32]), ids[:32], feats)[0][0]
    assert not np.array_equal(s, first32 + o.pool_points_csr(np.array([0, 68]), ids[32:], feats)[0][0])


def test_merge_apply_ref_equals_oracle_round():
    """One round of oracle_np.merge_graph accumulates merged sums exactly as merge_apply_ref restates them."""
    rng = np.random.default_rng(3)
    R, E, D = 3000, 9000, 20
    u = rng.integers(0, R, E)
    v = (u + rng.integers(1, R, E)) % R
    keys = np.unique(o.pack_keys(u, v))
    blen = rng.integers(1, 50, keys.size).astype(np.uint32)
    cnt = rng.integers(1, 6, R).astype(np.int32)
    sum_ = rng.standard_normal((R, D)).astype(np.float32)
    area = rng.integers(1, 1000, R).astype(np.int64)
    per = rng.integers(2000, 2100, R).astype(np.int64)
    scores = o.score_l2(o.region_mean(sum_, cnt), keys)
    tau = float(np.quantile(scores, 0.4))
    want = o.merge_graph(sum_, cnt, area, per, keys, blen, tau=tau, max_rounds=1)
    lo, hi = o.unpack_keys(keys)
    sel = scores < np.float32(tau)
    parent = o.min_root_propagate(R, lo[sel], hi[sel])
    assert np.bincount(parent).max() > 32                           # long runs of members
    got = merge_apply_ref(parent, np.ones(R, np.uint8), sum_, cnt, area, per)
    assert want["rounds"] == 1 and got["n_merged"] == want["merges"]
    assert np.array_equal(got["sum"].view(np.uint32), want["sum"].view(np.uint32))
    assert np.array_equal(got["cnt"], want["cnt"]) and np.array_equal(got["area"], want["area"])
    rev = merge_apply_ref(parent, np.ones(R, np.uint8), sum_, cnt, area, per, descending=True)
    assert not np.array_equal(rev["sum"], want["sum"])


# ------------------------------------------------------------------------------------------
# GPU: point pooling
# ------------------------------------------------------------------------------------------
def pool_passes(D):
    """K (groups of 32 columns) of every 128-column pass of pool_points_pass."""
    return [min(4, -(-min(D - d0, 128) // 32)) for d0 in range(0, D, 128)]


def pool_id(pts, D, pad, shuffled, wrap):
    Ks = pool_passes(D)
    return "pts%d-chunks%d-D%d-K%s-pass%d-%s-%s-%s" % (
        pts, -(-pts // 32), D, ".".join(map(str, Ks)), len(Ks), "ld%d" % (D + pad) if pad else "dense",
        "shuffled" if shuffled else "ascending", "wrap" if wrap else "onesweep")


# (points of the special regions, D, feat_ld - D, shuffled membership, R beyond one sweep of the warps)
POOL_CASES = [
    (0, 1, 0, False, False),
    (1, 31, 0, True, True),
    (3, 32, 5, False, False),
    (4, 33, 0, True, True),
    (5, 64, 3, True, False),
    (31, 65, 0, True, True),
    (32, 96, 7, False, True),
    (33, 97, 0, True, True),
    (33, 300, 20, True, False),
    (64, 128, 0, True, True),
    (64, 100, 4, False, True),
    (65, 129, 7, True, True),
    (65, 1, 0, True, False),
    (1000, 257, 3, True, True),
    (1000, 32, 0, False, False),
]


def pool_ranges(R):
    return {"interior": (R // 3, 2 * R // 3), "first": (0, 0), "last": (R - 1, R - 1), "all": (0, R - 1),
            "clamped": (-5, R + 5), "none": (INT64_MAX, -1), "reversed": (5, 4)}


@pytest.mark.gpu
@pytest.mark.parametrize("pts,D,pad,shuffled,wrap", [pytest.param(*c, id=pool_id(*c)) for c in POOL_CASES])
def test_pool_points_exact(cuda, pts, D, pad, shuffled, wrap):
    """dm_pool_points_csr, dm_pool_points_csr_mean (D <= 128) and dm_pool_points_csr_tile over every kind of region
    range, bit for bit against the sequential fp32 restatement; outside a range cnt is 0 and sum rows keep the
    sentinel."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    R = 2 * S * 64 + 77 if wrap else S * 32 + 7
    nw = warps_for(R, S)
    assert (R > nw) == wrap and (R > 2 * nw) == wrap                 # wrap: every warp looks ahead past the sweep
    rng = np.random.default_rng(1000 * pts + D + pad)
    specials = np.unique(np.r_[[x for x in (0, 1, R // 2, R - 2, R - 1, nw - 1, nw, nw + 1, 2 * nw + 5) if x < R],
                               rng.choice(R, 24, replace=False)])
    offsets, ids, wide = csr_inputs(rng, R, pts, specials, D, D + pad, shuffled)
    feats = wide[:, :D]
    cnt_np = np.diff(offsets)
    assert cnt_np.max() == max(pts, 5) and (cnt_np == 0).any()
    if shuffled:
        assert any((np.diff(ids[offsets[r]:offsets[r + 1]]) < 0).any() for r in specials[:8]) or pts < 2
    want_s, want_c, want_m, want_n2 = pool_ref(offsets, ids, feats)
    off_t, ids_t, f_t = T(offsets, cuda), T(ids, cuda), T(wide, cuda)
    ld = D + pad

    def fresh():
        return (torch.full((R, D), float(SENTINEL), dtype=torch.float32, device=cuda),
                torch.full((R,), -7, dtype=torch.int32, device=cuda))

    s, c = fresh()
    L.check(L.dm_pool_points_csr(off_t.data_ptr(), ids_t.data_ptr(), f_t.data_ptr(), ld, R, D, s.data_ptr(), c.data_ptr(),
                                 None), "dm_pool_points_csr")
    same(s.cpu().numpy(), want_s)
    assert np.array_equal(c.cpu().numpy(), want_c)
    if D <= 128:
        s, c = fresh()
        m = torch.full((R, D), float(SENTINEL), dtype=torch.float32, device=cuda)
        n2 = torch.full((R,), float(SENTINEL), dtype=torch.float32, device=cuda)
        L.check(L.dm_pool_points_csr_mean(off_t.data_ptr(), ids_t.data_ptr(), f_t.data_ptr(), ld, R, D, s.data_ptr(),
                                          c.data_ptr(), m.data_ptr(), n2.data_ptr(), None), "dm_pool_points_csr_mean")
        same(s.cpu().numpy(), want_s)
        assert np.array_equal(c.cpu().numpy(), want_c)
        same(m.cpu().numpy(), want_m)
        same(n2.cpu().numpy(), want_n2)
    for name, (a, b) in pool_ranges(R).items():
        rg = torch.tensor([a, b], dtype=torch.int64, device=cuda)
        s, c = fresh()
        L.check(L.dm_pool_points_csr_tile(off_t.data_ptr(), ids_t.data_ptr(), f_t.data_ptr(), ld, R, D, s.data_ptr(),
                                          c.data_ptr(), rg.data_ptr(), None), "dm_pool_points_csr_tile " + name)
        inside = np.zeros(R, bool)
        inside[max(a, 0):min(b, R - 1) + 1] = True
        gs, gc = s.cpu().numpy(), c.cpu().numpy()
        same(gs[inside], want_s[inside])
        assert np.array_equal(gc[inside], want_c[inside]), name
        assert (gc[~inside] == 0).all(), name
        assert (gs[~inside].view(np.uint32) == SENT_U32).all(), name
        assert inside.any() == (name not in ("none", "reversed"))


ID_RANGE_CASES = ["n0", "all-invalid", "beyond-R", "one-valid", "extremes-past-one-sweep"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ID_RANGE_CASES)
def test_points_id_range(cuda, case):
    """dm_points_id_range = (min, max) of the ids in [0, R), (INT64_MAX, -1) when there is none."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    R = 5000
    rng = np.random.default_rng(len(case))
    if case == "n0":
        rop = np.zeros(0, np.int32)
    elif case == "all-invalid":
        rop = np.full(3000, -1, np.int32)
    elif case == "beyond-R":
        rop = rng.integers(-1, R, 3000).astype(np.int32)
        rop[rng.choice(3000, 500, replace=False)] = rng.choice(np.array([R, R + 7, 2 ** 31 - 1], np.int32), 500)
    elif case == "one-valid":
        rop = np.array([-1, R, 17, -5, R + 1], np.int32)
    else:
        n = 2 * S * 4 * 256 + 99
        assert n > grid_for(n, S, 256, 4) * 256                     # threads stride over more than one sweep
        rop = rng.integers(R // 4, R // 2, n).astype(np.int32)
        rop[rng.choice(n, 1000, replace=False)] = -1
        rop[n - 1], rop[n - 40] = 3, R - 2                          # the extremes sit in the last sweep
    ok = (rop >= 0) & (rop < R)
    want = [int(rop[ok].min()), int(rop[ok].max())] if ok.any() else [INT64_MAX, -1]
    rg = torch.tensor([123, 456], dtype=torch.int64, device=cuda)
    rop_ptr = T(rop, cuda).data_ptr() if rop.size else None
    L.check(L.dm_points_id_range(rop_ptr, rop.size, R, rg.data_ptr(), None), "dm_points_id_range")
    assert rg.cpu().tolist() == want


# ------------------------------------------------------------------------------------------
# GPU: region means
# ------------------------------------------------------------------------------------------
MEAN_D = [1, 31, 33, 100, 128, 129, 260]


@pytest.mark.gpu
@pytest.mark.parametrize("D", MEAN_D, ids=["D%d-trips%d-wrap" % (D, -(-D // 128)) for D in MEAN_D])
def test_region_mean_exact(cuda, D):
    """dm_region_mean over every region (more regions than warps): IEEE division, FMA-chain norm; cnt == 0 gives
    NaN mean and NaN norm2 whatever the sum row holds."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    R = 2 * S * 64 + 77
    assert warps_for(R, S) < R
    rng = np.random.default_rng(D)
    sum_ = (rng.standard_normal((R, D)) * 5).astype(np.float32)
    cnt = rng.integers(0, 40, R).astype(np.int32)
    cnt[[0, R - 1]] = 0
    want_m = o.region_mean(sum_, cnt)
    want_n2 = norm2_ref(want_m)
    assert np.isnan(want_n2[cnt == 0]).all() and np.isfinite(want_n2[cnt > 0]).all()
    m = torch.full((R, D), float(SENTINEL), dtype=torch.float32, device=cuda)
    n2 = torch.full((R,), float(SENTINEL), dtype=torch.float32, device=cuda)
    s_t, c_t = T(sum_, cuda), T(cnt, cuda)
    L.check(L.dm_region_mean(s_t.data_ptr(), c_t.data_ptr(), R, D, m.data_ptr(), n2.data_ptr(), None, None),
            "dm_region_mean")
    same(m.cpu().numpy(), want_m)
    same(n2.cpu().numpy(), want_n2)


@pytest.mark.gpu
@pytest.mark.parametrize("D", MEAN_D, ids=["D%d-only-wrap" % D for D in MEAN_D])
def test_region_mean_only_exact(cuda, D):
    """dm_region_mean with `only`: a warp looks at 32 flags at a time and the sparse loop wraps past one sweep of
    nwarps * 32 regions.  Flagged rows equal the restatement, every other row of mean and norm2 keeps the sentinel."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    nw = S * 64
    R = nw * 32 + 1000
    assert warps_for(R, S) == nw and R > nw * 32
    g = torch.Generator(device=cuda).manual_seed(D)
    s_t = torch.randn((R, D), generator=g, device=cuda) * 5
    c_t = torch.randint(0, 40, (R,), generator=g, device=cuda, dtype=torch.int32)
    rng = np.random.default_rng(D)
    sw = nw * 32
    idx = np.unique(np.r_[[0, 31, 32, 33, R - 1, sw - 1, sw, sw + 31, sw + 32, sw + 33],
                          rng.choice(R, 300, replace=False)])
    c_t[T(idx[::7], cuda)] = 0                                       # flagged regions without points
    only = torch.zeros(R, dtype=torch.uint8, device=cuda)
    idx_t = T(idx, cuda)
    only[idx_t] = 1
    m = torch.full((R, D), float(SENTINEL), dtype=torch.float32, device=cuda)
    n2 = torch.full((R,), float(SENTINEL), dtype=torch.float32, device=cuda)
    L.check(L.dm_region_mean(s_t.data_ptr(), c_t.data_ptr(), R, D, m.data_ptr(), n2.data_ptr(), only.data_ptr(), None),
            "dm_region_mean")
    want_m = o.region_mean(s_t[idx_t].cpu().numpy(), c_t[idx_t].cpu().numpy())
    same(m[idx_t].cpu().numpy(), want_m)
    same(n2[idx_t].cpu().numpy(), norm2_ref(want_m))
    assert np.isnan(want_m[::7]).all()
    m[idx_t] = float(SENTINEL)
    n2[idx_t] = float(SENTINEL)
    assert bool((m.view(torch.int32) == SENT_I32).all()) and bool((n2.view(torch.int32) == SENT_I32).all())


# ------------------------------------------------------------------------------------------
# GPU: merged statistics
# ------------------------------------------------------------------------------------------
APPLY_SIZES = [2, 31, 32, 33, 64, 65, 1000]
# (D, largest component): a root with more than HUB_MAX_SORT members sends the member list's bucket sort to its radix path
APPLY_CASES = [(1, 1000), (7, 5000), (100, 1000), (100, 5000), (128, 5000), (129, 1000), (260, 5000), (260, 1000)]


def apply_id(D, big):
    return "D%d-cols%d-%s-max%d" % (D, -(-D // 128), "radix" if big > HUB_MAX_SORT else "bucket", big)


class ApplyState:
    """Device copies of the per-region state dm_merge_apply updates."""

    def __init__(self, cuda, parent, alive, sum_, cnt, area, perim):
        self.parent, self.alive, self.sum = T(parent.astype(np.int32), cuda), T(alive, cuda), T(sum_, cuda)
        self.cnt, self.area, self.perim = T(cnt, cuda), T(area, cuda), T(perim, cuda)

    def apply(self, L, cuda, root_mask=None, masked_entry=True):
        import torch
        R, D = self.sum.shape
        changed = torch.full((R,), 7, dtype=torch.uint8, device=cuda)
        nm = torch.full((1,), -1, dtype=torch.int64, device=cuda)
        wsb = L.dm_merge_apply_workspace_bytes(R)
        ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
        args = (self.parent.data_ptr(), self.alive.data_ptr(), changed.data_ptr(), self.sum.data_ptr(), self.cnt.data_ptr(),
                self.area.data_ptr(), self.perim.data_ptr(), R, D, nm.data_ptr())
        if masked_entry:
            L.check(L.dm_merge_apply_masked(*args, None if root_mask is None else T(root_mask, cuda).data_ptr(),
                                            ws.data_ptr(), wsb, None), "dm_merge_apply_masked")
        else:
            L.check(L.dm_merge_apply(*args, ws.data_ptr(), wsb, None), "dm_merge_apply")
        return dict(sum=self.sum.cpu().numpy(), cnt=self.cnt.cpu().numpy(), area=self.area.cpu().numpy(),
                    perim=self.perim.cpu().numpy(), alive=self.alive.cpu().numpy(), changed=changed.cpu().numpy(),
                    n_merged=int(nm.item()))


def check_apply(got, want):
    same(got["sum"], want["sum"])
    for k in ("cnt", "area", "perim", "alive", "changed"):
        assert np.array_equal(got[k], want[k]), k
    assert got["n_merged"] == want["n_merged"]


def uf_run(L, cuda, parent_t, keys, sel, n=None, cap=None):
    """dm_uf_union over the first n entries (default all), then dm_uf_compress."""
    import torch
    R = parent_t.shape[0]
    n = keys.size if n is None else n
    cap = keys.size if cap is None else cap
    keys_t = T(keys.view(np.int64), cuda)
    sel_t = T(sel.astype(np.uint8), cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    L.check(L.dm_uf_union(parent_t.data_ptr(), keys_t.data_ptr(), sel_t.data_ptr(), nd.data_ptr(), cap, None), "dm_uf_union")
    L.check(L.dm_uf_compress(parent_t.data_ptr(), R, None), "dm_uf_compress")


@pytest.mark.gpu
@pytest.mark.parametrize("D,big", [pytest.param(*c, id=apply_id(*c)) for c in APPLY_CASES])
def test_merge_apply_exact(cuda, D, big):
    """dm_merge_apply / _masked against merge_apply_ref: min-root components of 2 .. `big` members, a (root, member)
    list longer than one sweep of the summing warps, already-dead members that must not be counted again; with a
    root mask on half of the roots; and a second round (unions over roots, compress, apply) from the first one's
    state."""
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    R = 40000
    rng = np.random.default_rng(D + big)
    sizes = [s for s in APPLY_SIZES + [5000] if s <= big] + list(rng.integers(2, 7, 3000))
    parent = components(rng, R, sizes)
    alive = np.ones(R, np.uint8)
    members = np.nonzero(parent != np.arange(R))[0]
    dead = rng.choice(members, 300, replace=False)                  # absorbed earlier: parent moved on, not alive
    alive[dead] = 0
    alive[rng.choice(np.nonzero(parent == np.arange(R))[0], 50, replace=False)] = 0     # dead, parent[x] == x
    alive[parent] = 1                                               # every root is alive
    sum_ = rng.standard_normal((R, D)).astype(np.float32)
    cnt = rng.integers(0, 9, R).astype(np.int32)
    area = rng.integers(1, 10 ** 6, R).astype(np.int64)
    perim = rng.integers(4, 10 ** 5, R).astype(np.int64)
    want = merge_apply_ref(parent, alive, sum_, cnt, area, perim)
    assert want["n_merged"] > warps_for(R, S)                       # the list spans more than one sweep
    assert (np.bincount(parent[(alive != 0) & (parent != np.arange(R))]).max() > HUB_MAX_SORT) == (big > HUB_MAX_SORT)
    st = ApplyState(cuda, parent, alive, sum_, cnt, area, perim)
    check_apply(st.apply(L, cuda, masked_entry=False), want)

    # root mask on every other root: masked roots merge their sums, the others keep theirs; integers merge everywhere
    roots = np.unique(parent[(alive != 0) & (parent != np.arange(R))])
    mask = np.zeros(R, np.uint8)
    mask[roots[::2]] = 1
    want_m = merge_apply_ref(parent, alive, sum_, cnt, area, perim, root_mask=mask)
    assert np.array_equal(want_m["sum"][roots[1::2]], sum_[roots[1::2]])
    check_apply(ApplyState(cuda, parent, alive, sum_, cnt, area, perim).apply(L, cuda, root_mask=mask), want_m)

    # round 2: unite random pairs of roots, compress, apply again
    u, v = rng.choice(roots, 400), rng.choice(roots, 400)
    u, v = u[u != v], v[u != v]
    keys = o.pack_keys(np.minimum(u, v), np.maximum(u, v))
    uf_run(L, cuda, st.parent, keys, np.ones(keys.size, np.uint8))
    parent2 = o.min_root_propagate(R, np.r_[np.arange(R), u], np.r_[parent, v])
    assert np.array_equal(st.parent.cpu().numpy(), parent2)
    want2 = merge_apply_ref(parent2, want["alive"], want["sum"], want["cnt"], want["area"], want["perim"])
    assert want2["n_merged"] > 0
    check_apply(st.apply(L, cuda), want2)


# ------------------------------------------------------------------------------------------
# GPU: union-find
# ------------------------------------------------------------------------------------------
UF_CASES = ["star-hub0", "star-hublast", "chain-reversed", "duplicates", "random-2^20", "second-round",
            "count-below-capacity"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", UF_CASES)
def test_union_find_exact(cuda, case):
    """dm_uf_union + dm_uf_compress give every region the minimum id of its component (oracle_np.min_root_propagate):
    CAS contention on one hub, a deep chain hooked from its far end, repeated edges, a large random graph, a second
    round on a compressed forest, and a device count below the capacity whose selected tail must be ignored."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(len(case))
    pk = lambda a, b: o.pack_keys(np.minimum(a, b), np.maximum(a, b))
    rounds = []                                                      # (keys, selected, n, cap) per round
    if case.startswith("star"):
        R = (1 << 17) + 1
        hub = 0 if case == "star-hub0" else R - 1
        leaves = rng.permutation(np.setdiff1d(np.arange(R), [hub]))
        keys = pk(np.full(leaves.size, hub), leaves)
        rounds.append((keys, np.ones(keys.size, np.uint8), keys.size, keys.size))
    elif case == "chain-reversed":
        R = 1 << 17
        i = np.arange(R - 2, -1, -1)
        keys = pk(i, i + 1)
        rounds.append((keys, np.ones(keys.size, np.uint8), keys.size, keys.size))
    elif case == "duplicates":
        R = 50000
        u = rng.integers(0, R, 40000)
        v = (u + rng.integers(1, R, 40000)) % R
        keys = rng.permutation(np.tile(pk(u, v), 3))
        rounds.append((keys, (rng.random(keys.size) < 0.6).astype(np.uint8), keys.size, keys.size))
    elif case == "random-2^20":
        R, E = 1 << 20, 1 << 21
        u = rng.integers(0, R, E)
        v = (u + rng.integers(1, R, E)) % R
        keys = pk(u, v)
        rounds.append((keys, (rng.random(E) < 0.5).astype(np.uint8), E, E))
    elif case == "second-round":
        R = 1 << 16
        for _ in range(2):
            u = rng.integers(0, R, 40000)
            v = (u + rng.integers(1, R, 40000)) % R
            keys = pk(u, v)
            rounds.append((keys, (rng.random(keys.size) < 0.5).astype(np.uint8), keys.size, keys.size))
    else:
        R, n = 100000, 30000
        u = rng.integers(0, R, n)
        v = (u + rng.integers(1, R, n)) % R
        i = np.arange(R - 1)
        keys = np.r_[pk(u, v), pk(i, i + 1)]                        # the tail past n would join everything
        sel = np.r_[(rng.random(n) < 0.5).astype(np.uint8), np.ones(R - 1, np.uint8)]
        rounds.append((keys, sel, n, keys.size))
    parent_t = torch.arange(R, dtype=torch.int32, device=cuda)
    eu, ev = [], []
    for keys, sel, n, cap in rounds:
        uf_run(L, cuda, parent_t, keys, sel, n, cap)
        lo, hi = o.unpack_keys(keys[:n])
        s = sel[:n] != 0
        eu.append(lo[s])
        ev.append(hi[s])
        want = o.min_root_propagate(R, np.concatenate(eu), np.concatenate(ev))
        assert np.array_equal(parent_t.cpu().numpy(), want)
    assert want.min() == 0 and (np.unique(want).size > 1) == (case not in ("star-hub0", "star-hublast", "chain-reversed"))


# ------------------------------------------------------------------------------------------
# GPU: selection
# ------------------------------------------------------------------------------------------
SEL_N = {"1": lambda S: 1, "31": lambda S: 31, "33": lambda S: 33, "2sweeps+77": lambda S: 2 * S * 8 * 256 + 77}
SEL_KINDS = ["l2-tau0", "l2-tau0.5", "mlp-o2", "mlp-o3", "mlp-o16"]


@pytest.mark.gpu
@pytest.mark.parametrize("n_name", list(SEL_N))
@pytest.mark.parametrize("kind", SEL_KINDS)
def test_merge_select_exact(cuda, kind, n_name):
    """dm_merge_select_l2 flags score < tau (score == tau, -0.0 against 0, NaN and +inf are not selected, -inf is);
    dm_merge_select_mlp flags o[e, 1] > o[e, 0] and never looks at columns >= 2 (ties and NaN are not selected).
    Flags past the device count keep what they held, and the count is exact."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    n = SEL_N[n_name](S)
    cap = n + 1000
    assert (n > grid_for(cap, S) * 256) == (n_name == "2sweeps+77")
    rng = np.random.default_rng(n + len(kind))
    f32 = np.float32
    if kind.startswith("l2"):
        tau = f32(0.0 if kind == "l2-tau0" else 0.5)
        v = (rng.standard_normal(cap) * 0.5 + tau).astype(f32)
        special = np.array([tau, np.nextafter(tau, f32(-np.inf)), np.nextafter(tau, f32(np.inf)), f32(-0.0), f32(0.0),
                            f32(np.nan), f32(np.inf), f32(-np.inf)], f32)
        for j in range(special.size):                               # at both ends of the counted entries
            v[j % n] = special[j]
            v[n - 1 - (j % n)] = special[-1 - j]
        v[rng.choice(n, n // 50, replace=False)] = tau
        v[n:] = -np.inf                                              # past the count: would be selected
        want = v[:n] < tau
        v_t = T(v, cuda)
    else:
        n_out = int(kind[5:])
        v = rng.standard_normal((cap, n_out)).astype(f32)
        v[:, 2:] = np.where(rng.random((cap, n_out - 2)) < 0.5, f32(3e38), f32(np.inf))   # ignored columns
        pairs = [(1.0, 1.0), (0.0, -0.0), (-0.0, 0.0), (np.nan, 1.0), (1.0, np.nan), (np.nan, np.nan), (-np.inf, np.inf),
                 (np.inf, np.inf), (0.5, np.nextafter(f32(0.5), f32(1)))]
        for j, (a, b) in enumerate(pairs):
            for e in (j % n, n - 1 - (j % n)):
                v[e, 0], v[e, 1] = a, b
        tie = rng.choice(n, n // 50, replace=False)
        v[tie, 1] = v[tie, 0]
        v[n:, 0], v[n:, 1] = -np.inf, np.inf
        want = v[:n, 1] > v[:n, 0]
        v_t = T(v, cuda)
    assert n < 33 or (0 < want.sum() < n)
    sel = torch.full((cap,), 0xAB, dtype=torch.uint8, device=cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    ns = torch.full((1,), -1, dtype=torch.int64, device=cuda)
    if kind.startswith("l2"):
        L.check(L.dm_merge_select_l2(v_t.data_ptr(), float(tau), nd.data_ptr(), cap, sel.data_ptr(), ns.data_ptr(), None),
                "dm_merge_select_l2")
    else:
        L.check(L.dm_merge_select_mlp(v_t.data_ptr(), n_out, nd.data_ptr(), cap, sel.data_ptr(), ns.data_ptr(), None),
                "dm_merge_select_mlp")
    got = sel.cpu().numpy()
    assert np.array_equal(got[:n], want.astype(np.uint8))
    assert (got[n:] == 0xAB).all()
    assert int(ns.item()) == int(want.sum())


# ------------------------------------------------------------------------------------------
# GPU: re-keyed edge list
# ------------------------------------------------------------------------------------------
# (path, R, raw entries, distinct neighbours of region 0): the hashed run reduction with small buckets and with hub
# buckets; its radix fall-back for more hubs than the hub list holds (a shape of test_edges_sort_unique) and for one
# bucket above the hub limit
REKEY_CASES = [("hashed", 20000, 60000, 0), ("hashed-hubs", 700, 300000, 0), ("radix-hubcount", 2500, 2500000, 0),
               ("radix-hubsize", 20000, 60000, 5000)]


def rekey_path(unique_keys, R, cap):
    """sort_unique's choice for dm_edges_rekey (n_ids = R, key_bits = 2 id_bits): the hashed reduction when R <= 4 cap
    + 65536, unless a bucket (unique keys per low id) holds more than HUB_MAX or more than HUB_CAP buckets hold more
    than HUB_MIN."""
    if R > 4 * cap + 65536:
        return "radix"
    deg = np.bincount((unique_keys >> np.uint64(32)).astype(np.int64), minlength=R)
    if (deg > HUB_MAX).any():
        return "radix-hubsize"
    if (deg > HUB_MIN).sum() > HUB_CAP:
        return "radix-hubcount"
    return "hashed-hubs" if (deg > HUB_MIN).any() else "hashed"


@pytest.mark.gpu
@pytest.mark.parametrize("path,R,n,hub", [pytest.param(*c, id="%s-R%d-n%d" % c[:3]) for c in REKEY_CASES])
def test_edges_rekey_exact(cuda, path, R, n, hub):
    """dm_edges_rekey: keys (root(u), root(v)) sorted and unique, lengths summed, 2 len taken off the perimeter of the
    root of every edge that became internal, and each run carries the score of its first pair (lowest input index),
    on the hashed path and on its radix fall-back."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    rng = np.random.default_rng(R + n)
    u = rng.integers(0, R, n)
    v = (u + rng.integers(1, R, n)) % R
    parent = components(rng, R, list(rng.integers(2, 5, R // 10)))
    members = np.nonzero(parent != np.arange(R))[0]
    j = rng.choice(n, n // 20, replace=False)                       # edges that become internal
    u[j] = rng.choice(members, j.size)
    v[j] = parent[u[j]]
    u[:hub], v[:hub] = 0, rng.choice(np.arange(1, R), hub, replace=False)
    keys = o.pack_keys(np.minimum(u, v), np.maximum(u, v))
    lens = rng.integers(1, 1000, n).astype(np.uint32)
    scores = rng.standard_normal(n).astype(np.float32)
    perim = rng.integers(10 ** 6, 10 ** 7, R).astype(np.int64)
    lo, hi = o.unpack_keys(keys)
    a, b = parent[lo], parent[hi]
    loop = a == b
    idx = np.nonzero(~loop)[0]
    nk = o.pack_keys(np.minimum(a, b), np.maximum(a, b))[idx]
    uk, first, inv, runs = np.unique(nk, return_index=True, return_inverse=True, return_counts=True)
    want_len = np.bincount(inv, weights=lens[idx].astype(np.float64), minlength=uk.size).astype(np.uint32)
    want_score = scores[idx[first]]
    want_perim = perim.copy()
    np.add.at(want_perim, a[loop], -2 * lens[loop].astype(np.int64))
    assert loop.sum() > 0 and (runs > 1).sum() > 0
    cap = n + 33
    assert rekey_path(uk, R, cap) == path
    keys_t = torch.full((cap,), -1, dtype=torch.int64, device=cuda)
    keys_t[:n] = T(keys.view(np.int64), cuda)
    lens_t = torch.zeros(cap, dtype=torch.int32, device=cuda)
    lens_t[:n] = T(lens.view(np.int32), cuda)
    sc_t = torch.full((cap,), float(SENTINEL), dtype=torch.float32, device=cuda)
    sc_t[:n] = T(scores, cuda)
    nd = torch.tensor([n], dtype=torch.int64, device=cuda)
    parent_t, perim_t = T(parent.astype(np.int32), cuda), T(perim, cuda)
    wsb = L.dm_edges_rekey_workspace_bytes(cap)
    ws = torch.empty(wsb, dtype=torch.uint8, device=cuda)
    L.check(L.dm_edges_rekey(parent_t.data_ptr(), keys_t.data_ptr(), lens_t.data_ptr(), sc_t.data_ptr(), nd.data_ptr(), cap,
                             R, perim_t.data_ptr(), ws.data_ptr(), wsb, None), "dm_edges_rekey")
    m = int(nd.item())
    assert m == uk.size
    assert np.array_equal(keys_t[:m].cpu().numpy().view(np.uint64), uk)
    assert np.array_equal(lens_t[:m].cpu().numpy().view(np.uint32), want_len)
    same(sc_t[:m].cpu().numpy(), want_score)
    assert np.array_equal(perim_t.cpu().numpy(), want_perim)


# ------------------------------------------------------------------------------------------
# GPU: a row tile without sample points, end to end
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sharded_row_tile_without_points(cuda):
    """Three virtual ranks; the middle tile keeps no sample points, so its engine pools an empty region range
    ((INT64_MAX, -1) from dm_points_id_range).  The label map equals the oracle's and the single-GPU engine's on the
    same reduced set of points."""
    import torch
    from deepmerge_b200 import merge_scene
    from deepmerge_b200.sharded import ShardedMergeEngine, points_in_tile, tile_bounds
    world, H, W, R, tau = 3, 240, 384, 600, 0.5
    sc = o.synth_scene(H, W, R, C=4)
    n, D = sc["n_regions"], sc["feats"].shape[1]
    ym0, ym1 = tile_bounds(H, world, 1)
    keep = np.nonzero(~((sc["ys"] >= ym0) & (sc["ys"] < ym1)))[0]
    assert keep.size < sc["ys"].size
    xs, ys, feats = sc["xs"][keep], sc["ys"][keep], sc["feats"][keep]
    want = o.merge_scene(sc["labels"], n, sc["region_of_point"][keep], feats, tau=tau)
    assert want["merges"] > 0
    Tc = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(cuda)
    fd = FakeDist(world)
    results, errors = [None] * world, []

    def rank_main(rank):
        try:
            fd.local.rank = rank
            torch.cuda.set_device(cuda)
            y0, y1 = tile_bounds(H, world, rank)
            last = rank == world - 1
            mine = points_in_tile(torch.from_numpy(ys), y0, y1).numpy()
            eng = ShardedMergeEngine(H, W, n, D, 4, len(mine), fd, cuda)
            res = eng.run(Tc(sc["labels"][y0:y1 + (0 if last else 1)]), Tc(feats[mine]), tau,
                          image_tile=Tc(sc["image"][y0:y1]), xs_local=Tc(xs[mine]), ys_local_rel=Tc(ys[mine] - y0))
            torch.cuda.synchronize()
            results[rank] = (len(mine), eng.eng.id_range.cpu().tolist(), res.labels.cpu().numpy(), res.root.cpu().numpy(),
                             res.rounds, res.merges)
        except Exception as e:          # surface thread failures in the test
            errors.append(e)
            fd.bar.abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    assert results[1][0] == 0 and results[1][1] == [INT64_MAX, -1]
    assert all(r[0] > 0 and 0 <= r[1][0] <= r[1][1] < n for r in (results[0], results[2]))
    full = np.concatenate([r[2] for r in results])
    assert np.array_equal(full, want["labels"])
    for r in results:
        assert np.array_equal(r[3], want["root"]) and r[4] == want["rounds"] and r[5] == want["merges"]
    single = merge_scene(Tc(sc["labels"]), Tc(feats), tau, n_regions=n, image=Tc(sc["image"]), xs=Tc(xs), ys=Tc(ys))
    assert np.array_equal(single.labels.cpu().numpy(), full)
