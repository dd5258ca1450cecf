"""The exchange layer of the sharded merge loop compared exactly: rank visibility (dm_mark_endpoints, dm_shard_seen,
dm_shard_frontier), the frontier union-find (dm_shard_frontier_pairs, dm_uf_union_slots), the growth plan
(dm_shard_propagate, dm_shard_plan), the row slots (dm_rows_pack, dm_rows_unpack, dm_rows_unpack_slots,
dm_slots_overflow, dm_slots_word_max), the round flags (dm_shard_round_flags), the edge-list concatenation
(dm_edges_concat) and the peer kernels (dm_peer_put_slot, dm_peer_allreduce_i32), each against a numpy restatement of
its header text, plus dm_perimeter's handling of keys that are not edges.

Three layers:
  * every entry point alone, at the edges where it could go wrong: counts above capacity, garbage behind a count,
    sentinel and out-of-range ids, rank bits up to 30, and sizes on both sides of its grid-stride loop;
  * the frontier argument (one exchange of (shared component, local root) pairs plus one MIN all-reduce of parent gives
    the global min-id root, DESIGN.md "union-find by frontier exchange") played with W virtual ranks on one GPU, kernels
    only, with a numpy twin that shows which shortcuts the topologies catch;
  * ShardedMergeEngine on its peer transport (PeerSlots / PeerArray) with ranks emulated as threads and a stand-in for
    torch's symmetric memory, compared bit for bit with the collective transport and with the oracle.

Ranks that share one GPU run one after another on one stream; all cross-rank ordering is host synchronisation, and no
kernel waits on another.  Buffers that a wrong index could leave sit inside a larger allocation with guard bytes on
both sides, so a stray write shows as a changed guard.

Each GPU case asserts the path its inputs take, restating the grid rule grid_for of csrc/common.cuh: per-region kernels
(and dm_rows_pack, 256 regions per block) loop once the item count exceeds 2048 S, the one-warp-per-entry kernels once
it exceeds 64 S (S = dm_num_sms()); the test ids name the path.
"""
import threading
import types

import numpy as np
import pytest

from oracle import oracle_np as o
from test_gpu_scorers_exact import T, num_sms
from test_gpu_stats_exact import grid_for
from test_gpu_sharded import FakeDist

GUARD, FILL = 256, 0xA5                     # guard bytes on each side of a buffer under test, and their value
FILL32 = int(np.array([0xA5A5A5A5], np.uint32).view(np.int32)[0])
INT_MIN, INT_MAX = -2 ** 31, 2 ** 31 - 1


def lib():
    from deepmerge_b200._lib import lib as _l
    return _l()


# ------------------------------------------------------------------------------------------
# path rules (csrc/common.cuh grid_for; the launch of each entry point in csrc/merge.cu / csrc/rag.cu)
# ------------------------------------------------------------------------------------------
def item_loops(items, S):
    """A one-thread-per-item kernel launched with grid_for(items) blocks of 256 threads runs its loop more than once."""
    return items > grid_for(items, S) * 256


def warp_loops(entries, S):
    """A one-warp-per-entry kernel launched with grid_for(entries * 32) blocks of 8 warps runs its loop more than once."""
    return entries > grid_for(entries * 32, S) * 8


def path(loops):
    return "stride" if loops else "single"


# ------------------------------------------------------------------------------------------
# restatements of the header text
# ------------------------------------------------------------------------------------------
def pack(lo, hi):
    return (np.asarray(lo, np.uint64) << np.uint64(32)) | np.asarray(hi, np.uint64)


def unpack(k):
    k = np.asarray(k, np.uint64)
    return (k >> np.uint64(32)).astype(np.int64), (k & np.uint64(0xFFFFFFFF)).astype(np.int64)


def is_edge(keys, R):
    """Both ids of the key in [0, R), compared unsigned: the (R, R) sentinel and ~0 are not edges."""
    lo, hi = unpack(keys)
    return (lo < R) & (hi < R)


def mark_endpoints_ref(flags, keys, n, R):
    f = flags.copy()
    k = keys[:n][is_edge(keys[:n], R)]
    lo, hi = unpack(k)
    f[lo] = 1
    f[hi] = 1
    return f


def perimeter_ref(keys, lens, n, border, R):
    p = border.astype(np.int64).copy()
    ok = is_edge(keys[:n], R)
    lo, hi = unpack(keys[:n][ok])
    np.add.at(p, lo, lens[:n][ok].astype(np.int64))
    np.add.at(p, hi, lens[:n][ok].astype(np.int64))
    return p


def two_bits(m):
    m = np.asarray(m, np.int64)
    return (m & (m - 1)) != 0


def shard_seen_ref(area, seen, cnt, rank):
    sees = (seen != 0) | (area > 0)
    mask_cnt = np.r_[np.where(sees, 1 << rank, 0), cnt].astype(np.int32)
    return sees.astype(np.uint8), mask_cnt, cnt.copy()


def shard_frontier_ref(mask_cnt, cnt_local):
    R = cnt_local.shape[0]
    return mask_cnt[R:].copy(), (two_bits(mask_cnt[:R]) & (cnt_local > 0)).astype(np.uint8)


def frontier_pairs_ref(parent, alive, mask, rank):
    """(region, its local root) for every alive region seen here and elsewhere that is not its own root."""
    bit = 1 << rank
    R = parent.shape[0]
    m = mask.astype(np.int64)
    x = np.nonzero((alive != 0) & ((m & bit) != 0) & ((m & ~bit) != 0) & (parent != np.arange(R)))[0]
    return np.sort(pack(x, parent[x]))


def min_components(R, a, b):
    """Min-id label of every id of the undirected graph on [0, R) with edges (a[i], b[i])."""
    lab = np.arange(R, dtype=np.int64)
    a, b = np.asarray(a, np.int64), np.asarray(b, np.int64)
    while True:
        ra, rb = lab[a], lab[b]
        m = np.minimum(ra, rb)
        new = lab.copy()
        np.minimum.at(new, ra, m)                   # hook the larger label's representative under the smaller
        np.minimum.at(new, rb, m)
        while True:                                 # pointer jumping: new[x] <= x, so this ends
            nn = new[new]
            if np.array_equal(nn, new):
                break
            new = nn
        new = new[lab]
        if np.array_equal(new, lab) and np.array_equal(lab[a], lab[b]):
            return lab.astype(np.int32)
        lab = new


def forest_edges(parent):
    x = np.nonzero(parent != np.arange(parent.shape[0]))[0]
    return x, parent[x]


def propagate_ref(parent, alive, mask):
    R = parent.shape[0]
    mask, grew = mask.copy(), np.zeros(R, np.uint8)
    x = np.nonzero((alive != 0) & (parent != np.arange(R)))[0]
    np.bitwise_or.at(mask, parent[x], mask[x])
    grew[parent[x]] = 1
    return mask, grew


def plan_ref(parent, alive, mask_old, mask_new, grew, rank):
    bit = 1 << rank
    mo, mp = mask_old.astype(np.int64), mask_new[parent].astype(np.int64)
    seen_comp = ((mask_new.astype(np.int64) & bit) != 0).astype(np.uint8)
    send = (alive != 0) & (grew[parent] != 0) & two_bits(mp) & ((mo & -mo) == bit)
    return send.astype(np.uint8), seen_comp


def round_flags_ref(counts, flags, first_round):
    f = flags.copy()
    f[0] = counts[4]
    if first_round:
        f[3] = int(counts[2] != 0)
        f[4] = int(counts[3] == 1)
        f[6] = counts[1]
    if counts[3] > 1:
        f[5] = 1
    return f


def concat_ref(keys, lens, counts, slot_cap, dst_cap):
    parts_k = [keys[g * slot_cap:g * slot_cap + min(c, slot_cap)] for g, c in enumerate(counts)]
    parts_l = [lens[g * slot_cap:g * slot_cap + min(c, slot_cap)] for g, c in enumerate(counts)]
    k, ln = np.concatenate(parts_k), np.concatenate(parts_l)
    bad = int(any(c > slot_cap for c in counts) or k.shape[0] > dst_cap)
    return k[:dst_cap], ln[:dst_cap], min(k.shape[0], dst_cap), bad


def put_extent(n, cap, hdr, segs):
    """Byte ranges of a slot that dm_peer_put_slot stores: the header and, of each segment, min(n, cap) elements
    rounded up to whole 16-byte units."""
    n = min(n, cap)
    return [(0, hdr)] + [(off, off + -(-(n * elem) // 16) * 16) for off, elem in segs]


# ------------------------------------------------------------------------------------------
# device helpers
# ------------------------------------------------------------------------------------------
class Guarded:
    """nbytes of device memory with GUARD bytes of FILL on each side (one allocation); the region itself starts FILLed
    too unless init is given."""

    def __init__(self, cuda, nbytes, init=None):
        import torch
        self.n = int(nbytes)
        self.buf = torch.full((2 * GUARD + self.n,), FILL, dtype=torch.uint8, device=cuda)
        self.t = self.buf[GUARD:GUARD + self.n]
        if init is not None:
            b = np.ascontiguousarray(init).view(np.uint8).reshape(-1)
            assert b.shape[0] == self.n
            self.t.copy_(T(b, cuda))

    def ptr(self):
        return self.t.data_ptr()

    def get(self, dtype):
        return self.t.cpu().numpy().view(dtype)

    def intact(self):
        b = self.buf.cpu().numpy()
        return bool((b[:GUARD] == FILL).all() and (b[GUARD + self.n:] == FILL).all())


_ALIVE = []


def dptr(x, cuda):
    """Device address of a device copy of the numpy array x that stays allocated until the test ends (a temporary
    tensor would go back to the caching allocator before the launch, and the next input could take its block)."""
    t = T(x, cuda)
    _ALIVE.append(t)
    return t.data_ptr()


@pytest.fixture(autouse=True)
def _inputs_outlive_the_test():
    yield
    if _ALIVE:
        sync()
        _ALIVE.clear()


def dev_i64(cuda, v):
    return dptr(np.array([v], np.int64), cuda)


def sync():
    import torch
    torch.cuda.synchronize()


def random_forest(rng, R, n_comp, alive_frac=1.0):
    """Compressed min-root forest: n_comp components of random sizes over scattered ids; alive flags (roots alive)."""
    parent = np.arange(R, dtype=np.int32)
    perm = rng.permutation(R)
    cuts = np.sort(rng.choice(np.arange(1, R), size=min(n_comp, R - 1), replace=False))
    for grp in np.split(perm, cuts):
        if grp.size > 1 and rng.random() < 0.7:
            parent[grp] = grp.min()
    alive = (rng.random(R) < alive_frac).astype(np.uint8)
    alive[parent == np.arange(R)] = 1
    return parent, alive


def random_masks(rng, R, W_bits=31, max_bits=3):
    """int32 visibility masks with 0..max_bits bits among bits 0..W_bits-1 (bits 29 and 30 included)."""
    m = np.zeros(R, np.int64)
    for _ in range(max_bits):
        b = rng.integers(0, W_bits, R)
        m |= np.where(rng.random(R) < 0.5, np.int64(1) << b, 0)
    return m.astype(np.int32)


# ------------------------------------------------------------------------------------------
# CPU: the restatements
# ------------------------------------------------------------------------------------------
def test_restatement_helpers():
    keys = np.array([pack(1, 2), pack(5, 5), 2 ** 64 - 1, pack(7, 3), pack(2, 7)], np.uint64)
    assert is_edge(keys, 5).tolist() == [True, False, False, False, False]
    assert is_edge(keys, 8).tolist() == [True, True, False, True, True]
    f = mark_endpoints_ref(np.zeros(8, np.uint8), keys, 4, 8)
    assert f.tolist() == [0, 1, 1, 1, 0, 1, 0, 1]
    p = perimeter_ref(keys, np.array([1, 10, 100, 1000, 5], np.uint32), 5, np.zeros(8, np.int64), 8)
    assert p.tolist() == [0, 1, 6, 1000, 0, 20, 0, 1005]
    assert put_extent(5, 4, 16, [(16, 4), (32, 12)]) == [(0, 16), (16, 32), (32, 80)]
    assert put_extent(3, 8, 80, [(80, 8), (80, 0)]) == [(0, 80), (80, 112), (80, 80)]
    assert two_bits(np.array([0, 1, 2, 3, 1 << 30, (1 << 30) | 1])).tolist() == [False, False, False, True, False, True]


def test_min_components_against_python_union_find():
    rng = np.random.default_rng(0)
    for R, E in ((1, 0), (10, 3), (500, 400), (3000, 2900)):
        a, b = rng.integers(0, R, E), rng.integers(0, R, E)
        p = list(range(R))

        def find(x):
            while p[x] != x:
                x = p[x]
            return x
        for x, y in zip(a, b):
            rx, ry = find(int(x)), find(int(y))
            if rx != ry:
                p[max(rx, ry)] = min(rx, ry)
        want = np.array([find(x) for x in range(R)], np.int32)
        assert np.array_equal(min_components(R, a, b), want)
    chain = np.arange(2000)[::-1]                   # a long path in adversarial order
    assert (min_components(2000, chain[:-1], chain[1:]) == 0).all()


def test_plan_and_frontier_restatements_follow_their_rules():
    """Hand-worked cases of the rules the kernels implement: the lowest bit of mask_old[x], two bits of the component's
    new mask, a dead or unshared region sends nothing; a pair needs this rank's bit and another one."""
    parent = np.array([0, 0, 0, 3, 3], np.int32)
    alive = np.array([1, 1, 0, 1, 1], np.uint8)
    mask_old = np.array([1, 6, 1, 1 << 30, 1 << 30], np.int32)
    mask_new = np.array([7, 6, 1, 1 << 30, 1 << 30], np.int32)
    grew = np.array([1, 0, 0, 1, 0], np.uint8)
    send, seen = plan_ref(parent, alive, mask_old, mask_new, grew, 1)
    assert send.tolist() == [0, 1, 0, 0, 0] and seen.tolist() == [1, 1, 0, 0, 0]
    send, _ = plan_ref(parent, alive, mask_old, mask_new, grew, 0)
    assert send.tolist() == [1, 0, 0, 0, 0]                  # region 2 is dead
    send, _ = plan_ref(parent, alive, mask_old, mask_new, grew, 30)
    assert send.tolist() == [0, 0, 0, 0, 0]                  # component 3 is seen by one rank only
    mask = np.array([3, 3, 3, 1, (1 << 30) | 1], np.int32)
    got = frontier_pairs_ref(parent, alive, mask, 0)
    assert got.tolist() == [int(pack(1, 0)), int(pack(4, 3))]   # 0 is a root, 2 dead, 3 a root
    assert frontier_pairs_ref(parent, alive, mask, 30).tolist() == [int(pack(4, 3))]


# ------------------------------------------------------------------------------------------
# GPU: endpoints and perimeter -- keys that are not edges
# ------------------------------------------------------------------------------------------
def bad_keys(R):
    return np.array([2 ** 64 - 1, pack(R, R), pack(R + 3, 1), pack(2, R + 5)], np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("R,n,cap", [pytest.param(50, 0, 40, id="single-n0"), pytest.param(1000, 300, 700, id="single-garbage"),
                                     pytest.param(5000, 5000, 5000, id="single-full"),
                                     pytest.param(None, None, None, id="stride-garbage")])
def test_mark_endpoints_exact(request, cuda, R, n, cap):
    """flags[lo] = flags[hi] = 1 for the first n keys (read on the device) that are edges: entries behind n are in-range
    garbage that must stay unread, ~0 / (R, R) / out-of-range keys are skipped, preset flags stay set, and nothing is
    written outside flags."""
    L, S = lib(), num_sms()
    if R is None:
        cap = 2048 * S + 333
        R, n = cap + 17, cap - 5
    assert request.node.callspec.id.startswith(path(n > grid_for(cap, S) * 256))     # the grid is sized by capacity
    rng = np.random.default_rng(R + n)
    lo = rng.integers(0, R, cap)
    hi = rng.integers(0, R, cap)
    keys = pack(np.minimum(lo, hi), np.maximum(lo, hi))
    sl = rng.choice(n, size=min(n, 8), replace=False) if n else []
    keys[sl] = np.resize(bad_keys(R), len(sl))
    flags0 = (rng.random(R) < 0.05).astype(np.uint8)
    fl = Guarded(cuda, R, flags0)
    L.check(L.dm_mark_endpoints(dptr(keys.view(np.int64), cuda), dev_i64(cuda, n), cap, R, fl.ptr(), None),
            "dm_mark_endpoints")
    want = mark_endpoints_ref(flags0, keys, n, R)
    assert fl.intact()
    assert np.array_equal(fl.get(np.uint8), want)
    if n < cap:
        assert not np.array_equal(mark_endpoints_ref(flags0, keys, cap, R), want)     # the garbage would show


@pytest.mark.gpu
def test_mark_endpoints_skips_keys_that_are_not_edges(cuda):
    """~0 (the default sentinel of the graph primitives), (R, R) and keys with an id >= R mark nothing: flags sits
    between guards, and a key whose id reads as -1 or >= R through a signed compare would write into them."""
    L = lib()
    R = 64
    keys = np.r_[bad_keys(R), pack(3, 9)].astype(np.uint64)
    fl = Guarded(cuda, R, np.zeros(R, np.uint8))
    L.check(L.dm_mark_endpoints(dptr(keys.view(np.int64), cuda), dev_i64(cuda, keys.shape[0]),
                                keys.shape[0], R, fl.ptr(), None), "dm_mark_endpoints")
    sync()
    assert fl.intact(), "dm_mark_endpoints wrote outside flags"
    assert np.nonzero(fl.get(np.uint8))[0].tolist() == [3, 9]


@pytest.mark.gpu
def test_perimeter_skips_keys_that_are_not_edges(cuda):
    """dm_perimeter: border + lengths of incident edges; ~0, (R, R) and out-of-range keys add nothing anywhere."""
    L = lib()
    R = 64
    rng = np.random.default_rng(5)
    lo, hi = rng.integers(0, R, 200), rng.integers(0, R, 200)
    keys = np.r_[bad_keys(R), pack(np.minimum(lo, hi), np.maximum(lo, hi))].astype(np.uint64)
    rng.shuffle(keys)
    lens = rng.integers(1, 1000, keys.shape[0]).astype(np.uint32)
    border = rng.integers(0, 50, R).astype(np.int64)
    pm = Guarded(cuda, 8 * R)
    L.check(L.dm_perimeter(dptr(keys.view(np.int64), cuda), dptr(lens.view(np.int32), cuda),
                           dev_i64(cuda, keys.shape[0]), keys.shape[0], dptr(border, cuda), pm.ptr(), R,
                           None), "dm_perimeter")
    sync()
    assert pm.intact(), "dm_perimeter wrote outside perimeter"
    assert np.array_equal(pm.get(np.int64), perimeter_ref(keys, lens, keys.shape[0], border, R))


# ------------------------------------------------------------------------------------------
# GPU: visibility and counts
# ------------------------------------------------------------------------------------------
def region_sizes(S):
    return [("single", 1000), ("single", 2048 * S - 1), ("stride", 2048 * S + 777)]


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [0, 1, 29, 30])
@pytest.mark.parametrize("size", [0, 2], ids=["single", "stride"])
def test_shard_seen_and_frontier_exact(cuda, rank, size):
    """dm_shard_seen: seen |= area > 0, mask half = my bit where seen, count half and cnt_local = cnt.  dm_shard_frontier:
    cnt = the count half, send = the mask has two bits and cnt_local > 0 (not != 0)."""
    L, S = lib(), num_sms()
    p, R = region_sizes(S)[size]
    assert path(item_loops(R, S)) == p
    rng = np.random.default_rng(rank * 7 + size)
    area = np.where(rng.random(R) < 0.4, 0, rng.integers(1, 10 ** 6, R)).astype(np.int64)
    seen = (rng.random(R) < 0.3).astype(np.uint8)
    cnt = rng.integers(-3, 50, R).astype(np.int32)
    sg = Guarded(cuda, R, seen)
    mc = Guarded(cuda, 8 * R)
    cl = Guarded(cuda, 4 * R)
    L.check(L.dm_shard_seen(dptr(area, cuda), sg.ptr(), dptr(cnt, cuda), rank, R, mc.ptr(), cl.ptr(), None),
            "dm_shard_seen")
    w_seen, w_mc, w_cl = shard_seen_ref(area, seen, cnt, rank)
    assert sg.intact() and mc.intact() and cl.intact()
    assert np.array_equal(sg.get(np.uint8), w_seen)
    assert np.array_equal(mc.get(np.int32), w_mc) and np.array_equal(cl.get(np.int32), w_cl)
    # the frontier on masks as the all-reduce leaves them: several ranks' bits, counts summed over ranks
    mask_cnt = np.r_[random_masks(rng, R), rng.integers(0, 100, R)].astype(np.int32)
    cnt_local = rng.integers(-2, 3, R).astype(np.int32)
    cg = Guarded(cuda, 4 * R)
    snd = Guarded(cuda, R)
    L.check(L.dm_shard_frontier(dptr(mask_cnt, cuda), dptr(cnt_local, cuda), R, cg.ptr(), snd.ptr(), None),
            "dm_shard_frontier")
    w_cnt, w_send = shard_frontier_ref(mask_cnt, cnt_local)
    assert cg.intact() and snd.intact()
    assert np.array_equal(cg.get(np.int32), w_cnt) and np.array_equal(snd.get(np.uint8), w_send)
    assert w_send.any() and (two_bits(mask_cnt[:R]) & (cnt_local < 0)).any()       # the > 0 rule is exercised


# ------------------------------------------------------------------------------------------
# GPU: frontier pairs and their union
# ------------------------------------------------------------------------------------------
FLAG_WORDS = np.arange(101, 109, dtype=np.int64)


def fslot_bytes(cap):
    b = 80 + 8 * cap
    return b + (-b) % 16


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [0, 1, 29, 30])
@pytest.mark.parametrize("size,over", [(0, False), (0, True), (2, False), (2, True)],
                         ids=["single", "single-overflow", "stride", "stride-overflow"])
def test_frontier_pairs_exact(cuda, rank, size, over):
    """The pair set (order is atomic: compared sorted) and the count.  Dead, unshared and root regions send nothing.
    With count > capacity the first capacity slots hold distinct true pairs and nothing is written past them.  Only the
    16-byte count is cleared: the eight flag words behind it keep the caller's values."""
    L, S = lib(), num_sms()
    p, R = region_sizes(S)[size]
    assert path(item_loops(R, S)) == p
    rng = np.random.default_rng(100 + rank + size)
    parent, alive = random_forest(rng, R, R // 4, alive_frac=0.8)
    mask = random_masks(rng, R)
    mask[rng.random(R) < 0.3] |= np.int32(1 << rank)
    want = frontier_pairs_ref(parent, alive, mask, rank)
    n = want.shape[0]
    cap = n // 2 if over else n + 10
    cap += cap % 2
    nb = fslot_bytes(cap)
    init = np.full(nb, 0x5A, np.uint8)
    init[:8] = np.array([12345], np.int64).view(np.uint8)
    init[16:80] = FLAG_WORDS.view(np.uint8)
    sl = Guarded(cuda, nb, init)
    L.check(L.dm_shard_frontier_pairs(dptr(parent, cuda), dptr(alive, cuda), dptr(mask, cuda), rank,
                                      R, sl.ptr(), cap, None), "dm_shard_frontier_pairs")
    got = sl.get(np.uint8)
    assert sl.intact()
    assert got[:16].view(np.int64).tolist() == [n, 0]
    assert np.array_equal(got[16:80].view(np.int64), FLAG_WORDS)
    pairs = got[80:80 + 8 * cap].view(np.uint64)
    assert (got[80 + 8 * cap:] == 0x5A).all()
    if over:
        assert n > cap and np.unique(pairs).shape[0] == cap and np.isin(pairs, want).all()
    else:
        assert np.array_equal(np.sort(pairs[:n]), want)
        assert (pairs[n:].view(np.uint8) == 0x5A).all()
    # what the rules exclude is present in the input
    bit, ids = 1 << rank, np.arange(R)
    m = mask.astype(np.int64)
    shared = ((m & bit) != 0) & ((m & ~bit) != 0)
    assert (shared & (alive == 0) & (parent != ids)).any() and (shared & (parent == ids)).any()
    assert (((m & bit) != 0) & ~shared & (parent != ids)).any()


def union_slots_buffer(rng, n_slots, cap, counts, pair_lists, garbage_R):
    """Gathered frontier slots: [count | pad | 8 flag words | pairs[cap]] each; entries past a slot's count (and past
    cap) are in-range garbage pairs that would join components if read."""
    sb = fslot_bytes(cap)
    buf = np.zeros((n_slots, sb), np.uint8)
    for g in range(n_slots):
        buf[g, :8] = np.array([counts[g]], np.int64).view(np.uint8)
        buf[g, 16:80] = FLAG_WORDS.view(np.uint8)
        gar = pack(rng.integers(0, garbage_R, cap), rng.integers(0, garbage_R, cap))
        pl = pair_lists[g][:cap]
        gar[:pl.shape[0]] = pl
        buf[g, 80:80 + 8 * cap] = gar.view(np.uint8)
    return buf, sb


def used_pairs(pair_lists, counts, cap, R):
    ks = [pl[:max(0, min(c, cap))] for pl, c in zip(pair_lists, counts)]
    k = np.concatenate(ks) if ks else np.zeros(0, np.uint64)
    a, b = unpack(k)
    ok = (a < R) & (b < R)
    return a[ok], b[ok]


UNION_CASES = [(1, 64, "plain"), (2, 64, "chain"), (7, 100, "over"), (16, 64, "under"), (31, 50, "chain"),
               (31, 40, "bad-ids"), (31, None, "stride")]


@pytest.mark.gpu
@pytest.mark.parametrize("n_slots,cap,kind", [pytest.param(*c, id="%dslots-%s" % (c[0], c[2])) for c in UNION_CASES])
def test_uf_union_slots_exact(cuda, n_slots, cap, kind):
    """dm_uf_union_slots + dm_uf_compress = the min-id components of the local forest and the first min(count, cap)
    pairs of every slot whose ids are both < R.  Chains run across slots in adversarial order; count > cap uses only cap
    pairs; entries behind a smaller count are garbage that would merge components."""
    L, S = lib(), num_sms()
    R = 3000
    if cap is None:
        cap = -(-(2048 * S + 500) // n_slots)
        cap += cap % 2
        R = 200000
    items = n_slots * cap
    assert path(item_loops(items, S)) == ("stride" if kind == "stride" else "single")
    rng = np.random.default_rng(n_slots * 1000 + cap)
    parent, _ = random_forest(rng, R, R // 3)
    counts = [cap] * n_slots
    lists = []
    if kind == "chain":                              # one path through ids in random order, its links dealt across slots
        ids = rng.permutation(R)[:n_slots * cap]
        links = pack(ids[1:], ids[:-1])[::-1]
        for g in range(n_slots):
            lists.append(links[g::n_slots])
        counts = [lst.shape[0] for lst in lists]
    else:
        for g in range(n_slots):
            k = rng.integers(0, R, (cap + 20, 2))
            lists.append(pack(k[:, 0], k[:, 1]))
        if kind == "over":
            counts = [cap + 20] * n_slots
        elif kind == "under":
            counts = [int(c) for c in rng.integers(0, cap, n_slots)]
        elif kind == "bad-ids":
            for lst in lists:
                lst[::5] = pack(rng.integers(R, 2 ** 32, lst[::5].shape[0]), rng.integers(0, R, lst[::5].shape[0]))
                lst[1::7] = pack(rng.integers(0, R, lst[1::7].shape[0]), np.uint64(2 ** 32 - 1))
    buf, sb = union_slots_buffer(rng, n_slots, cap, counts, lists, R)
    a, b = used_pairs(lists, counts, cap, R)
    fa, fb = forest_edges(parent)
    want = min_components(R, np.r_[fa, a], np.r_[fb, b])
    pg = Guarded(cuda, 4 * R, parent)
    L.check(L.dm_uf_union_slots(pg.ptr(), dptr(buf, cuda), n_slots, sb, cap, R, None), "dm_uf_union_slots")
    L.check(L.dm_uf_compress(pg.ptr(), R, None), "dm_uf_compress")
    assert pg.intact()
    assert np.array_equal(pg.get(np.int32), want)
    if kind in ("over", "under"):                    # what the count excludes would change the result
        every = used_pairs([lst[:cap] for lst in lists], [cap] * n_slots, cap, R) if kind == "under" else \
            used_pairs(lists, [cap + 20] * n_slots, cap + 20, R)
        assert not np.array_equal(min_components(R, np.r_[fa, every[0]], np.r_[fb, every[1]]), want)


# ------------------------------------------------------------------------------------------
# GPU: growth plan
# ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("rank", [0, 30])
@pytest.mark.parametrize("size", [0, 2], ids=["single", "stride"])
def test_shard_propagate_and_plan_exact(cuda, rank, size):
    """dm_shard_propagate clears grew on every call and ORs the masks of alive absorbed regions into their root (dead
    members do not propagate); dm_shard_plan ships x when its component grew, is seen by two ranks and the lowest bit of
    mask_old[x] is this rank's -- the root itself included."""
    L, S = lib(), num_sms()
    p, R = region_sizes(S)[size]
    assert path(item_loops(R, S)) == p
    rng = np.random.default_rng(300 + rank + size)
    parent, alive = random_forest(rng, R, R // 5, alive_frac=0.7)
    mask = random_masks(rng, R, max_bits=2)
    lowest = rng.random(R) < 0.3
    mask[lowest] = (mask[lowest] & ~np.int32((1 << rank) - 1)) | np.int32(1 << rank)   # rank is the lowest bit here
    mg = Guarded(cuda, 4 * R, mask)
    gr = Guarded(cuda, R, (rng.random(R) < 0.5).astype(np.uint8))              # stale flags of an earlier round
    pt, at = T(parent, cuda), T(alive, cuda)
    L.check(L.dm_shard_propagate(pt.data_ptr(), at.data_ptr(), mg.ptr(), gr.ptr(), R, None), "dm_shard_propagate")
    w_mask, w_grew = propagate_ref(parent, alive, mask)
    assert mg.intact() and gr.intact()
    assert np.array_equal(mg.get(np.int32), w_mask) and np.array_equal(gr.get(np.uint8), w_grew)
    assert not np.array_equal(propagate_ref(parent, np.ones(R, np.uint8), mask)[0], w_mask)   # dead members matter
    snd, sc = Guarded(cuda, R), Guarded(cuda, R)
    L.check(L.dm_shard_plan(pt.data_ptr(), at.data_ptr(), dptr(mask, cuda), dptr(w_mask, cuda),
                            dptr(w_grew, cuda), rank, R, snd.ptr(), sc.ptr(), None), "dm_shard_plan")
    w_send, w_seen = plan_ref(parent, alive, mask, w_mask, w_grew, rank)
    assert snd.intact() and sc.intact()
    assert np.array_equal(snd.get(np.uint8), w_send) and np.array_equal(sc.get(np.uint8), w_seen)
    roots = parent == np.arange(R)
    assert (w_send.astype(bool) & roots).any() and (w_send.astype(bool) & ~roots).any()
    m_new_p = w_mask[parent].astype(np.int64)                   # the lowest bit of the component's mask is not the rule
    alt = (alive != 0) & (w_grew[parent] != 0) & two_bits(m_new_p) & ((m_new_p & -m_new_p) == (1 << rank))
    assert not np.array_equal(alt.astype(np.uint8), w_send)


# ------------------------------------------------------------------------------------------
# GPU: row slots
# ------------------------------------------------------------------------------------------
PACK_CASES = [(1000, 1, False), (999, 31, False), (1001, 32, False), (777, 33, False), (1000, 100, False),
              (513, 128, False), (1000, 129, False), (1000, 33, True), (None, 1, False), (None, 33, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("R,D,over", [pytest.param(*c, id="%s-D%d%s" % ("R%d" % c[0] if c[0] else "wrap", c[1],
                                                                        "-overflow" if c[2] else "")) for c in PACK_CASES])
def test_rows_pack_exact(cuda, R, D, over):
    """dm_rows_pack: the (id, row) set of the flagged regions, sorted by id, and their count; a count above capacity
    fills exactly capacity distinct entries and writes nothing past them."""
    L, S = lib(), num_sms()
    if R is None:
        R = 2048 * S + 1111
    assert R % 32 != 0
    assert path(item_loops(R, S)) == ("stride" if R > 2048 * S else "single")
    rng = np.random.default_rng(R + D)
    flag = (rng.random(R) < 0.2).astype(np.uint8)
    flag[[0, R - 1]] = 1
    rows = rng.standard_normal((R, D)).astype(np.float32)
    n = int(flag.sum())
    cap = n // 3 if over else n + 5
    ids_g, rows_g = Guarded(cuda, 4 * cap), Guarded(cuda, 4 * cap * D)
    n_out = Guarded(cuda, 8)
    L.check(L.dm_rows_pack(dptr(flag, cuda), dptr(rows, cuda), R, D, ids_g.ptr(), rows_g.ptr(), cap,
                           n_out.ptr(), None), "dm_rows_pack")
    assert ids_g.intact() and rows_g.intact() and n_out.intact()
    assert int(n_out.get(np.int64)[0]) == n
    ids = ids_g.get(np.int32)
    out = rows_g.get(np.float32).reshape(cap, D)
    k = min(n, cap)
    o_ = np.argsort(ids[:k])
    got_ids, got_rows = ids[:k][o_], out[:k][o_]
    if over:
        assert np.unique(got_ids).shape[0] == k and flag[got_ids].all()
    else:
        assert np.array_equal(got_ids, np.nonzero(flag)[0])
        assert (ids[k:].view(np.uint32) == 0xA5A5A5A5).all()
    assert np.array_equal(got_rows.view(np.uint32), rows[got_ids].view(np.uint32))


def unpack_ref(ids, in_rows, n, cap, R, rows, add):
    rows = rows.copy()
    for i in range(min(n, cap)):
        r = int(ids[i])
        if 0 <= r < R:
            rows[r] = rows[r] + in_rows[i] if add else in_rows[i]
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("add", [0, 1], ids=["copy", "add"])
@pytest.mark.parametrize("entries,over", [("below", False), ("above", False), ("above", True)],
                         ids=["single", "stride", "stride-overflow"])
def test_rows_unpack_exact(cuda, add, entries, over):
    """dm_rows_unpack: rows[id] = row, or rows[id] + row as one fp32 addition (bits compared); ids -1 and >= R are
    skipped; a count above capacity is clamped (the entries behind capacity hold valid ids that must stay unread)."""
    L, S = lib(), num_sms()
    D, R = 33, 200000
    cap = 64 * S - 7 if entries == "below" else 64 * S + 700
    assert path(warp_loops(cap, S)) == ("single" if entries == "below" else "stride")
    rng = np.random.default_rng(cap + add)
    ids = rng.permutation(R)[:cap + 100].astype(np.int32)
    ids[5::50] = -1
    ids[7::50] = R + rng.integers(0, 1000, ids[7::50].shape[0])
    in_rows = rng.standard_normal((cap + 100, D)).astype(np.float32)
    n = cap + 100 if over else cap - 3
    rows0 = rng.standard_normal((R, D)).astype(np.float32)
    rg = Guarded(cuda, 4 * R * D, rows0)
    L.check(L.dm_rows_unpack(dptr(ids, cuda), dptr(in_rows, cuda), dev_i64(cuda, n), cap, R, D,
                             rg.ptr(), add, None), "dm_rows_unpack")
    want = unpack_ref(ids, in_rows, n, cap, R, rows0, add)
    assert rg.intact()
    got = rg.get(np.float32).reshape(R, D)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def row_slots(rng, n_slots, cap, D, counts, R, ids_all):
    """Gathered row slots [count | pad | ids[cap] | rows[cap][D]]; ids_all[g] has cap ids (entries past the count are
    valid ids too)."""
    sb = 16 + 4 * cap * (D + 1)
    sb += (-sb) % 16
    buf = np.zeros((n_slots, sb), np.uint8)
    rows = rng.standard_normal((n_slots, cap, D)).astype(np.float32)
    for g in range(n_slots):
        buf[g, :8] = np.array([counts[g]], np.int64).view(np.uint8)
        buf[g, 16:16 + 4 * cap] = ids_all[g].astype(np.int32).view(np.uint8)
        buf[g, 16 + 4 * cap:16 + 4 * cap * (D + 1)] = rows[g].view(np.uint8).reshape(-1)
    return buf, sb, rows


@pytest.mark.gpu
@pytest.mark.parametrize("zero", [0, 1], ids=["copy", "zero"])
@pytest.mark.parametrize("entries", ["below", "above"], ids=["single", "stride"])
def test_rows_unpack_slots_exact(cuda, zero, entries):
    """dm_rows_unpack_slots: for every slot, entries below min(count, cap) copy (or clear) their row; ids -1 and >= R are
    skipped; entries behind a slot's count hold valid ids and must stay unread.  Counts above cap are clamped."""
    L, S = lib(), num_sms()
    D, R, n_slots = 33, 150000, 5
    total = 64 * S - 20 if entries == "below" else 64 * S + 900
    cap = -(-total // n_slots)
    assert path(warp_loops(n_slots * cap, S)) == ("single" if entries == "below" else "stride")
    rng = np.random.default_rng(total + zero)
    perm = rng.permutation(R)[:n_slots * cap].astype(np.int32)
    ids_all = perm.reshape(n_slots, cap).copy()
    ids_all[:, 3::40] = -1
    ids_all[:, 9::40] = R + 5
    counts = [cap, cap // 2, 0, cap + 50, cap - 1]
    buf, sb, srows = row_slots(rng, n_slots, cap, D, counts, R, ids_all)
    rows0 = rng.standard_normal((R, D)).astype(np.float32)
    rg = Guarded(cuda, 4 * R * D, rows0)
    L.check(L.dm_rows_unpack_slots(dptr(buf, cuda), n_slots, sb, cap, R, D, rg.ptr(), zero, None),
            "dm_rows_unpack_slots")
    want = rows0.copy()
    for g in range(n_slots):
        for i in range(min(counts[g], cap)):
            r = int(ids_all[g, i])
            if 0 <= r < R:
                want[r] = 0 if zero else srows[g, i]
    assert rg.intact()
    assert np.array_equal(rg.get(np.float32).reshape(R, D).view(np.uint32), want.view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("n_slots", [1, 63, 64, 65, 4096])
def test_slots_overflow_exact(cuda, n_slots):
    """flag = 1 when some slot's count exceeds capacity (the slot is anywhere, past the 64-thread block too); a flag that
    is already 1 stays 1, one that is 0 stays 0 when nothing overflows."""
    L = lib()
    sb, cap = 32, 100
    for where in [None, 0, n_slots - 1]:
        for pre in (0, 1):
            buf = np.zeros((n_slots, sb), np.uint8)
            counts = np.full(n_slots, cap, np.int64)
            counts[::3] = 0
            if where is not None:
                counts[where] = cap + 1
            buf[:, :8] = counts.view(np.uint8).reshape(n_slots, 8)
            buf[:, 8:16] = np.full(n_slots, 10 ** 9, np.int64).view(np.uint8).reshape(n_slots, 8)   # not a count
            fl = Guarded(cuda, 8, np.array([pre], np.int64))
            L.check(L.dm_slots_overflow(dptr(buf, cuda), n_slots, sb, cap, fl.ptr(), None), "dm_slots_overflow")
            assert fl.intact()
            assert int(fl.get(np.int64)[0]) == (1 if (pre or where is not None) else 0), (where, pre)


@pytest.mark.gpu
@pytest.mark.parametrize("n_slots", [0, 1, 31, 33, 4096])
def test_slots_word_max_exact(cuda, n_slots):
    """out = max over the slots of the int64 word at each offset the loop uses (0 for no slot); the maximum is placed in
    a slot of every lane group of the butterfly, and values above 2^32 keep their high half."""
    L = lib()
    sb = 48
    rng = np.random.default_rng(n_slots)
    for off in range(0, sb, 8):
        places = [None] if n_slots == 0 else sorted({0, n_slots - 1, min(n_slots - 1, 20), min(n_slots - 1, 17),
                                                      n_slots // 2})
        for place in places:
            words = rng.integers(0, 2 ** 40, (max(n_slots, 1), sb // 8)).astype(np.int64)[:n_slots]
            if place is not None:
                words[place, off // 8] = 2 ** 41 + place
            buf = np.ascontiguousarray(words).view(np.uint8)
            out = Guarded(cuda, 8, np.array([-7], np.int64))
            src = T(buf if n_slots else np.zeros(16, np.uint8), cuda)
            L.check(L.dm_slots_word_max(src.data_ptr(), n_slots, sb, off, out.ptr(), None), "dm_slots_word_max")
            want = int(words[:, off // 8].max()) if n_slots else 0
            assert out.intact()
            assert int(out.get(np.int64)[0]) == want, (off, place)


@pytest.mark.gpu
def test_shard_round_flags_table(cuda):
    """Every flag word for first_round 0 / 1 and counts[3] in {0, 1, 2}: [0] = selected every round; first round only
    [3] overflow, [4] bad label, [6] raw entries; [5] internal error any round; the rest keep their value; the slot
    header receives the same eight words."""
    L = lib()
    for first in (0, 1):
        for c3 in (0, 1, 2):
            for c2 in (0, 5):
                counts = np.array([11, 12345, c2, c3, 77, 99, 98, 97], np.int64)
                flags0 = np.array([-1, -2, -3, -4, -5, 0, -7, -8], np.int64)
                fl = Guarded(cuda, 64, flags0)
                sf = Guarded(cuda, 64)
                L.check(L.dm_shard_round_flags(dptr(counts, cuda), fl.ptr(), first, sf.ptr(), None),
                        "dm_shard_round_flags")
                want = round_flags_ref(counts, flags0, first)
                assert fl.intact() and sf.intact()
                assert fl.get(np.int64).tolist() == want.tolist(), (first, c3, c2)
                assert sf.get(np.int64).tolist() == want.tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("counts,slot_cap,dst_cap", [([3, 0, 5, 2], 6, 24), ([6, 9, 1], 6, 24), ([5, 5, 5, 5], 6, 12),
                                                     ([4, 7], 6, 100), ([2, 3], 6, 4), ([0, 0, 0], 6, 10)],
                         ids=["plain", "slot-over", "dst-over", "slot-over-only", "partial", "empty"])
def test_edges_concat_exact(cuda, counts, slot_cap, dst_cap):
    """dm_edges_concat keeps slot order; a slot count above slot_cap (clamped) and a total above dst_cap each set
    n_out[1]; the partial copy up to dst_cap is exact and nothing is written past it."""
    L = lib()
    rng = np.random.default_rng(slot_cap + dst_cap + sum(counts))
    n_lists = len(counts)
    keys = rng.integers(0, 2 ** 62, n_lists * slot_cap).astype(np.uint64)
    lens = rng.integers(1, 2 ** 31, n_lists * slot_cap).astype(np.uint32)
    dk, dl = Guarded(cuda, 8 * dst_cap), Guarded(cuda, 4 * dst_cap)
    n_out = Guarded(cuda, 16, np.array([-1, -1], np.int64))
    L.check(L.dm_edges_concat(dptr(keys.view(np.int64), cuda), dptr(lens.view(np.int32), cuda),
                              dptr(np.array(counts, np.int64), cuda), n_lists, slot_cap, dk.ptr(), dl.ptr(), dst_cap,
                              n_out.ptr(), None), "dm_edges_concat")
    wk, wl, tot, bad = concat_ref(keys, lens, counts, slot_cap, dst_cap)
    assert dk.intact() and dl.intact() and n_out.intact()
    assert n_out.get(np.int64).tolist() == [tot, bad]
    assert np.array_equal(dk.get(np.uint64)[:tot], wk) and np.array_equal(dl.get(np.uint32)[:tot], wl)
    assert (dk.get(np.uint8)[8 * tot:] == FILL).all() and (dl.get(np.uint8)[4 * tot:] == FILL).all()


# ------------------------------------------------------------------------------------------
# GPU: peer kernels, every rank's buffer on one device
# ------------------------------------------------------------------------------------------
PUT_LAYOUTS = {"rows": lambda cap, D: (16, [(16, 4), (16 + 4 * cap, 4 * D)]), "pairs": lambda cap, D: (80, [(80, 8), (80, 0)])}


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 8, 9, 31])
@pytest.mark.parametrize("layout", ["rows", "pairs"])
def test_peer_put_slot_exact(cuda, world, layout):
    """world gathered buffers on one device; ranks put one after another on one stream (the slices are disjoint, so
    this is the concurrent run's result).  Slot r of every buffer equals rank r's source over the header and the used
    part of each segment rounded up to 16 bytes; every other byte -- past that, and the slots of ranks that did not put
    -- keeps its fill.  Counts above capacity are clamped; a segment of element size 0 carries nothing."""
    import torch
    L = lib()
    cap, D = 24, 3                                      # segment offsets are multiples of 16
    hdr, segs = PUT_LAYOUTS[layout](cap, D)
    sb = max(off + cap * e for off, e in segs)
    sb += (-sb) % 16 + 16
    rng = np.random.default_rng(world * 10 + len(layout))
    bufs = [Guarded(cuda, world * sb) for _ in range(world)]
    bases = T(np.array([b.ptr() for b in bufs], np.int64), cuda)
    putters = [r for r in range(world) if world == 1 or r % 4 != 1]
    srcs, ns = {}, {}
    for r in putters:
        n = [5, 0, 1, 3, cap, cap + 9][r % 6]
        src = rng.integers(0, 255, sb).astype(np.uint8)
        src[:8] = np.array([n], np.int64).view(np.uint8)
        srcs[r], ns[r] = src, n
        st = T(src, cuda)
        L.check(L.dm_peer_put_slot(st.data_ptr(), bases.data_ptr(), world, r, sb, hdr, segs[0][0], segs[0][1], segs[1][0],
                                   segs[1][1], cap, None), "dm_peer_put_slot")
        torch.cuda.current_stream().synchronize()      # src is freed at the end of the iteration
    for p, b in enumerate(bufs):
        assert b.intact(), p
        got = b.get(np.uint8).reshape(world, sb)
        for r in range(world):
            want = np.full(sb, FILL, np.uint8)
            if r in srcs:
                for a, e in put_extent(ns[r], cap, hdr, segs):
                    want[a:e] = srcs[r][a:e]
            assert np.array_equal(got[r], want), (p, r)
    if layout == "rows":                                # the rounding matters: odd counts end inside a 16-byte unit
        assert any((min(n, cap) * 4) % 16 for n in ns.values())


def allreduce_ref(arrays, op):
    a = np.stack(arrays).astype(np.int64)
    if op:
        return a.min(0).astype(np.int32)
    return (a.sum(0) & 0xFFFFFFFF).astype(np.uint32).view(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 8, 9, 16, 17, 31, 64])
@pytest.mark.parametrize("op", [0, 1], ids=["sum", "min"])
def test_peer_allreduce_i32_exact(cuda, world, op):
    """Ranks reduce their slices one after another on one stream (disjoint slices: the concurrent run's result).  Every
    copy must equal the sum (wrapping int32) or the min, for n4 below world (empty slices), n4 not a multiple of world
    and larger arrays; the array sits at offset_bytes > 0 of each buffer and the words around it are guards.  min sees
    INT_MIN and INT_MAX; sum sees 31-bit masks with distinct bits per rank, whose sum is the OR."""
    L = lib()
    rng = np.random.default_rng(world * 2 + op)
    for n4 in sorted({max(1, world // 3), world + 1, 3 * world + 2, 1000}):
        n = 4 * n4
        off = 48
        arrays = []
        for r in range(world):
            if op:
                a = rng.integers(INT_MIN, INT_MAX, n, endpoint=True).astype(np.int32)
                a[rng.random(n) < 0.05] = INT_MAX
                a[rng.random(n) < 0.02] = INT_MIN
            elif world <= 31:
                a = np.where(rng.random(n) < 0.5, 1 << r, 0).astype(np.int32)
            else:
                a = rng.integers(INT_MIN, INT_MAX, n, endpoint=True).astype(np.int32)
            arrays.append(a)
        bufs = []
        for a in arrays:
            init = np.full(off // 4 + n + 8, FILL32, np.int32)
            init[off // 4:off // 4 + n] = a
            bufs.append(Guarded(cuda, 4 * init.shape[0], init))
        bases = T(np.array([b.ptr() for b in bufs], np.int64), cuda)
        for r in range(world):
            L.check(L.dm_peer_allreduce_i32(bases.data_ptr(), world, r, off, n, op, None), "dm_peer_allreduce_i32")
        want = allreduce_ref(arrays, op)
        if not op and world <= 31:
            assert np.array_equal(want, np.bitwise_or.reduce(np.stack(arrays), 0))
        for p, b in enumerate(bufs):
            got = b.get(np.int32)
            assert b.intact() and (got[:off // 4] == FILL32).all() and (got[off // 4 + n:] == FILL32).all(), (n4, p)
            assert np.array_equal(got[off // 4:off // 4 + n], want), (n4, p)


# ------------------------------------------------------------------------------------------
# the frontier argument with W virtual ranks
# ------------------------------------------------------------------------------------------
class Topology:
    """A global graph: edges (a, b, tile), the tile that sees each region, an optional start forest (round 2)."""

    def __init__(self):
        self.comps = []                    # (n_nodes, [(i, j, tile)], extra {node: tiles}, min node or None)

    def add(self, n, edges, extra=None, min_node=None):
        self.comps.append((n, edges, extra or {}, min_node))

    def build(self, rng, W, dead=0):
        N = sum(c[0] for c in self.comps)
        R = N + dead
        if dead:          # alive regions: id 0 and N - 1 others; every other id is a dead member of a smaller alive id
            node_ids = rng.permutation(np.r_[0, rng.choice(np.arange(1, R), N - 1, replace=False)])
        else:
            node_ids = rng.permutation(R)
        edges, mask = [], np.zeros(R, np.int64)
        pos = 0
        for n, es, extra, mn in self.comps:
            mine = node_ids[pos:pos + n].copy()
            if mn is not None:                           # the component's minimum id sits on the chosen node
                k = np.argmin(mine)
                mine[k], mine[mn] = mine[mn], mine[k]
            for i, j, t in es:
                edges.append((mine[i], mine[j], t))
                mask[mine[i]] |= 1 << t
                mask[mine[j]] |= 1 << t
            for i, ts in extra.items():
                for t in ts:
                    mask[mine[i]] |= 1 << t
            pos += n
        parent, alive = np.arange(R, dtype=np.int32), np.ones(R, np.uint8)
        if dead:
            alive_ids = np.sort(node_ids)
            for d in np.setdiff1d(np.arange(R), node_ids):
                cand = alive_ids[alive_ids < d]
                parent[d] = rng.choice(cand)
                alive[d] = 0
                mask[d] = rng.integers(0, 1 << W)          # a dead region's mask is stale: it must not matter
        return R, np.array(edges, np.int64).reshape(-1, 3), mask.astype(np.int32), parent, alive


def snake(topo, W, per_tile=3):
    """A path that crosses every tile and comes back; its minimum on an unshared node of tile 0's first visit."""
    tiles = list(range(W)) + list(range(W - 1, -1, -1))
    es = []
    for k, t in enumerate(tiles):
        for u in range(per_tile):
            i = k * per_tile + u
            es.append((i, i + 1, t))
    topo.add(len(tiles) * per_tile + 1, es, min_node=1)


def hub(topo, W, rng):
    es = []
    for t in range(W):
        es += [(0, 1 + 2 * t, t), (1 + 2 * t, 2 + 2 * t, t)]
    topo.add(1 + 2 * W, es, min_node=int(rng.integers(0, 1 + 2 * W)))


def root_shared(topo, W, rng):
    t = int(rng.integers(0, W - 1))
    topo.add(5, [(0, 1, t), (1, 2, t), (0, 3, t + 1), (3, 4, t + 1)], min_node=0)


def in_tile(topo, W, rng):
    n = int(rng.integers(2, 8))
    t = int(rng.integers(0, W))
    topo.add(n, [(int(rng.integers(0, i)), i, t) for i in range(1, n)], min_node=int(rng.integers(0, n)))


def singletons(topo, W, rng, k):
    for _ in range(k):
        topo.add(1, [], extra={0: [int(rng.integers(0, W))]})


TOPOLOGIES = ["snake", "hub", "root-shared", "in-tile", "round2"]


def make_topology(kind, W, seed):
    rng = np.random.default_rng(seed)
    topo = Topology()
    if kind in ("snake", "round2"):
        for _ in range(3):
            snake(topo, W)
    if kind in ("hub", "round2"):
        for _ in range(4):
            hub(topo, W, rng)
    if kind in ("root-shared", "round2"):
        for _ in range(6):
            root_shared(topo, W, rng)
    if kind in ("in-tile", "round2"):
        for _ in range(20):
            in_tile(topo, W, rng)
    singletons(topo, W, rng, 30)
    return topo.build(rng, W, dead=150 if kind == "round2" else 0)


def global_roots(R, edges, parent0):
    fa, fb = forest_edges(parent0)
    return min_components(R, np.r_[edges[:, 0], fa], np.r_[edges[:, 1], fb])


def frontier_twin(R, W, edges, mask, parent0, alive, exchange=True, allreduce=True, drop=None):
    """numpy twin of the virtual-rank procedure: local unions, frontier pairs, union of the gathered pairs, MIN."""
    parents, pairs = [], []
    for g in range(W):
        eg = edges[edges[:, 2] == g]
        fa, fb = forest_edges(parent0)
        p = min_components(R, np.r_[eg[:, 0], fa], np.r_[eg[:, 1], fb])
        parents.append(p)
        pairs.append(unpack(frontier_pairs_ref(p, alive, mask, g)))
    out = []
    for g in range(W):
        use = [pairs[h] for h in range(W) if h != drop] if exchange else [pairs[g]]
        fa, fb = forest_edges(parents[g])
        a = np.concatenate([fa] + [u[0] for u in use])
        b = np.concatenate([fb] + [u[1] for u in use])
        out.append(min_components(R, a, b))
    if allreduce:
        m = np.minimum.reduce(out)
        out = [m] * W
    return out


@pytest.mark.parametrize("W", [2, 3, 8, 9])
@pytest.mark.parametrize("kind", TOPOLOGIES)
def test_frontier_twin_gives_global_roots(W, kind):
    R, edges, mask, parent0, alive = make_topology(kind, W, W * 31 + len(kind))
    want = global_roots(R, edges, parent0)
    for p in frontier_twin(R, W, edges, mask, parent0, alive):
        assert np.array_equal(p, want)


@pytest.mark.parametrize("W", [3, 8, 9])
def test_frontier_twin_variants_are_caught(W):
    """Each shortcut gives a wrong parent on these topologies: no MIN all-reduce; uniting only the rank's own pairs (a
    snake over three or more tiles); dropping the pairs of the rank that holds the global minimum of a snake, whose
    unshared members two tiles away then never learn it."""
    wrong = lambda ps, want: any(not np.array_equal(p, want) for p in ps)
    for kind in TOPOLOGIES:
        R, edges, mask, parent0, alive = make_topology(kind, W, W * 31 + len(kind))
        want = global_roots(R, edges, parent0)
        assert wrong(frontier_twin(R, W, edges, mask, parent0, alive, allreduce=False), want), kind
        if kind in ("snake", "round2"):
            assert wrong(frontier_twin(R, W, edges, mask, parent0, alive, exchange=False), want), kind
            assert wrong(frontier_twin(R, W, edges, mask, parent0, alive, drop=0), want), kind


def virtual_ranks(cuda, R, W, edges, mask, parent0, alive):
    """The frontier union-find of one round with W ranks on one GPU, library kernels only: local dm_uf_union +
    dm_uf_compress, dm_shard_frontier_pairs, dm_peer_put_slot into W gathered buffers, dm_uf_union_slots +
    dm_uf_compress, dm_peer_allreduce_i32(min) over the W parent arrays.  Returns every rank's parent."""
    import torch
    L = lib()
    n_pad = R + (-R) % 4
    p0 = np.r_[parent0, np.arange(R, n_pad)].astype(np.int32)
    parents = [T(p0, cuda) for _ in range(W)]
    cap = R + R % 2
    sb = fslot_bytes(cap)
    slots = [torch.zeros(sb, dtype=torch.uint8, device=cuda) for _ in range(W)]
    gathered = [torch.zeros(W * sb, dtype=torch.uint8, device=cuda) for _ in range(W)]
    gbases = T(np.array([g.data_ptr() for g in gathered], np.int64), cuda)
    pbases = T(np.array([p.data_ptr() for p in parents], np.int64), cuda)
    at, mt = T(alive, cuda), T(mask, cuda)
    keep = []
    for g in range(W):
        eg = edges[edges[:, 2] == g]
        keys = pack(np.minimum(eg[:, 0], eg[:, 1]), np.maximum(eg[:, 0], eg[:, 1]))
        kt = T(np.r_[keys, np.zeros(1, np.uint64)].view(np.int64), cuda)
        sel = torch.ones(kt.shape[0], dtype=torch.uint8, device=cuda)
        nd = dev_i64(cuda, keys.shape[0])
        keep += [kt, sel]
        L.check(L.dm_uf_union(parents[g].data_ptr(), kt.data_ptr(), sel.data_ptr(), nd, kt.shape[0], None),
                "dm_uf_union")
        L.check(L.dm_uf_compress(parents[g].data_ptr(), R, None), "dm_uf_compress")
        L.check(L.dm_shard_frontier_pairs(parents[g].data_ptr(), at.data_ptr(), mt.data_ptr(), g, R, slots[g].data_ptr(), cap,
                                          None), "dm_shard_frontier_pairs")
    for g in range(W):
        L.check(L.dm_peer_put_slot(slots[g].data_ptr(), gbases.data_ptr(), W, g, sb, 80, 80, 8, 80, 0, cap, None),
                "dm_peer_put_slot")
    for g in range(W):
        L.check(L.dm_uf_union_slots(parents[g].data_ptr(), gathered[g].data_ptr(), W, sb, cap, R, None), "dm_uf_union_slots")
        L.check(L.dm_uf_compress(parents[g].data_ptr(), R, None), "dm_uf_compress")
    for g in range(W):
        L.check(L.dm_peer_allreduce_i32(pbases.data_ptr(), W, g, 0, n_pad, 1, None), "dm_peer_allreduce_i32")
    sync()
    return [p.cpu().numpy()[:R] for p in parents]


@pytest.mark.gpu
@pytest.mark.parametrize("W", [2, 3, 8, 9])
@pytest.mark.parametrize("kind", TOPOLOGIES)
def test_virtual_ranks_frontier_union_find(cuda, W, kind):
    """Every rank's parent after one exchange of frontier pairs and one MIN all-reduce equals the min-id components of
    the global graph, and equals the numpy twin's."""
    R, edges, mask, parent0, alive = make_topology(kind, W, W * 31 + len(kind))
    want = global_roots(R, edges, parent0)
    got = virtual_ranks(cuda, R, W, edges, mask, parent0, alive)
    for g, p in enumerate(got):
        assert np.array_equal(p, want), g


# ------------------------------------------------------------------------------------------
# the peer transport of ShardedMergeEngine, ranks emulated as threads
# ------------------------------------------------------------------------------------------
class PeerFakeDist(FakeDist):
    """FakeDist with the process group name the symmetric-memory rendezvous is keyed by."""
    group = types.SimpleNamespace(WORLD=types.SimpleNamespace(group_name="emulated"))


class FakeSymmetricMemory:
    """Stand-in for torch.distributed._symmetric_memory on one GPU: empty() is a plain allocation; the k-th rendezvous
    of every rank meets the other ranks' k-th, and its handle carries their data_ptr()s in rank order; barrier() is a
    device synchronisation followed by a host barrier of all ranks."""

    def __init__(self, fd):
        self.fd, self.lock, self.meetings = fd, threading.Lock(), {}

    def empty(self, *size, dtype=None, device=None):
        import torch
        return torch.empty(*size, dtype=dtype, device=device)

    def rendezvous(self, t, group_name):
        fd = self.fd
        k = getattr(fd.local, "n_rdv", 0)
        fd.local.n_rdv = k + 1
        with self.lock:
            meet = self.meetings.setdefault(k, [None] * fd.world)
        meet[fd.local.rank] = t
        fd.bar.wait()
        return types.SimpleNamespace(buffer_ptrs=[m.data_ptr() for m in meet], barrier=self.barrier)

    def barrier(self):
        import torch
        torch.cuda.synchronize()
        self.fd.bar.wait()


def run_sharded(cuda, monkeypatch, sc, world, tau, peer, mlp_w=None, row_capacity=None, gather=True):
    """ShardedMergeEngine on every rank of `world` threads, on the peer transport or the collective one.  Returns
    per-rank results (or the error strings when row_capacity is set)."""
    import torch
    import torch.distributed._symmetric_memory as symm
    from deepmerge_b200 import sharded
    from deepmerge_b200.sharded import ShardedMergeEngine, points_in_tile, tile_bounds
    H, W = sc["labels"].shape
    n, D = sc["n_regions"], sc["feats"].shape[1]
    fd = PeerFakeDist(world)
    fake = FakeSymmetricMemory(fd)
    monkeypatch.setattr(sharded, "_peer_exchange_possible", lambda dist: peer)
    monkeypatch.setattr(symm, "empty", fake.empty)
    monkeypatch.setattr(symm, "rendezvous", fake.rendezvous)
    results, errors = [None] * world, []

    def rank_main(rank):
        try:
            fd.local.rank = rank
            torch.cuda.set_device(cuda)
            y0, y1 = tile_bounds(H, world, rank)
            last = rank == world - 1
            mine = points_in_tile(torch.from_numpy(sc["ys"]), y0, y1).numpy()
            eng = ShardedMergeEngine(H, W, n, D, 4, len(mine), fd, cuda, row_capacity=row_capacity)
            eng.eng.use_graphs = False                   # host barriers across threads cannot sit inside a capture
            mlp = None
            if mlp_w is not None:
                from deepmerge_b200 import PackedMLP
                mlp = PackedMLP(*[T(w, cuda) for w in mlp_w])
            res = eng.run(T(sc["labels"][y0:y1 + (0 if last else 1)], cuda), T(sc["feats"][mine], cuda), tau,
                          image_tile=T(sc["image"][y0:y1], cuda), xs_local=T(sc["xs"][mine], cuda),
                          ys_local_rel=T(sc["ys"][mine] - y0, cuda), gather_outputs=gather, mlp=mlp)
            torch.cuda.synchronize()
            assert (eng.peer_rows is not None) == peer and (eng.peer_parent is not None) == peer
            results[rank] = dict(labels=res.labels.cpu().numpy(), root=res.root.cpu().numpy(), rounds=res.rounds,
                                 merges=res.merges, area=res.area.cpu().numpy(), perim=res.perimeter.cpu().numpy(),
                                 keys=res.edge_keys.cpu().numpy().view(np.uint64),
                                 bsum=eng.eng.bsum.cpu().numpy().view(np.uint64),
                                 sum=res.sum.cpu().numpy().view(np.uint32), cnt=res.cnt.cpu().numpy(),
                                 mask=eng.mask.cpu().numpy())
        except RuntimeError as e:
            errors.append(str(e))
            if row_capacity is None:
                fd.bar.abort()
        except BaseException as e:                       # surface thread failures in the test
            errors.append("unexpected: %r" % (e,))
            fd.bar.abort()

    threads = [threading.Thread(target=rank_main, args=(r,)) for r in range(world)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    monkeypatch.undo()
    if row_capacity is not None:
        return errors
    assert not errors, errors
    return results


def assert_same_ranks(a, b):
    """Everything bit for bit, the fp32 sums of the rows every rank holds included."""
    for ra, rb in zip(a, b):
        for k in ra:
            if isinstance(ra[k], np.ndarray):
                assert ra[k].shape == rb[k].shape and np.array_equal(ra[k], rb[k]), k
            else:
                assert ra[k] == rb[k], k


def assert_oracle(res, sc, want):
    full = np.concatenate([r["labels"] for r in res])
    assert np.array_equal(full, want["labels"])
    roots = np.unique(want["root"])
    for r in res:
        assert np.array_equal(r["root"], want["root"]) and r["rounds"] == want["rounds"] and r["merges"] == want["merges"]
        assert np.array_equal(r["area"][roots], want["area"][roots])
        assert np.array_equal(r["perim"][roots], want["perim"][roots])
        assert np.array_equal(r["keys"], want["keys"])


@pytest.mark.gpu
@pytest.mark.parametrize("world,H,W,R", [(2, 260, 384, 500), (3, 301, 640, 1500), (8, 301, 640, 1500), (9, 301, 640, 1500)])
def test_peer_transport_equals_collectives_and_oracle(cuda, monkeypatch, world, H, W, R):
    sc = o.synth_scene(H, W, R, C=4)
    want = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], tau=0.5)
    peer = run_sharded(cuda, monkeypatch, sc, world, 0.5, True)
    coll = run_sharded(cuda, monkeypatch, sc, world, 0.5, False)
    assert_same_ranks(peer, coll)
    assert_oracle(peer, sc, want)
    assert want["merges"] > 0 and any(two_bits(r["mask"]).any() for r in peer)


@pytest.mark.gpu
def test_peer_transport_cascade_three_rounds(cuda, monkeypatch):
    """The multi-round workload: the round body's exchange buffers are reused round after round."""
    from deepmerge_b200.synth import CASCADE_TAU
    H, W, R = 600, 800, 4000
    sc = o.synth_scene(H, W, R, C=4)
    sc["feats"] = o.synth_cascade_feats(sc["region_of_point"], sc["region_obj"], H, W, R)
    want = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], tau=CASCADE_TAU)
    assert want["rounds"] == 3
    peer = run_sharded(cuda, monkeypatch, sc, 3, CASCADE_TAU, True)
    coll = run_sharded(cuda, monkeypatch, sc, 3, CASCADE_TAU, False)
    assert_same_ranks(peer, coll)
    assert_oracle(peer, sc, want)


def hand_made_mlp(D):
    """The "same object?" network of the smoke test and the NCCL worker: logit 0 = L1 distance of the two pooled
    embeddings, logit 1 = 4, wide margins."""
    W1 = np.zeros((2 * D, 2 * D), np.float32)
    for d in range(D):
        W1[d, d], W1[d, D + d] = 1, -1
        W1[D + d, d], W1[D + d, D + d] = -1, 1
    W3 = np.zeros((2, 2 * D), np.float32)
    W3[0] = 1.0
    return [W1, np.zeros(2 * D, np.float32), np.eye(2 * D, dtype=np.float32), np.zeros(2 * D, np.float32), W3,
            np.array([0.0, 4.0], np.float32)]


@pytest.mark.gpu
def test_peer_transport_mlp_scored_loop(cuda, monkeypatch):
    """run(mlp=...) with the pair-MLP as the scorer at W = 3, on both transports: equal to each other and to the oracle."""
    H, W, R = 400, 512, 900
    sc = o.synth_scene(H, W, R, C=4)
    Wm = hand_made_mlp(sc["feats"].shape[1])
    want = o.merge_scene(sc["labels"], sc["n_regions"], sc["region_of_point"], sc["feats"], mlp=tuple(Wm))
    peer = run_sharded(cuda, monkeypatch, sc, 3, 0.0, True, mlp_w=Wm)
    coll = run_sharded(cuda, monkeypatch, sc, 3, 0.0, False, mlp_w=Wm)
    assert_same_ranks(peer, coll)
    assert want["merges"] > 0
    assert_oracle(peer, sc, want)


@pytest.mark.gpu
def test_peer_transport_row_slot_overflow_is_reported(cuda, monkeypatch):
    """A row slot too small for the exchange overflows on the peer path too: the stored count is clamped, the header
    keeps the true count, and every rank raises."""
    sc = o.synth_scene(120, 256, 400, C=4)
    errors = run_sharded(cuda, monkeypatch, sc, 2, 0.5, True, row_capacity=2)
    assert len(errors) == 2 and all("row exchange slot overflow" in e for e in errors), errors
