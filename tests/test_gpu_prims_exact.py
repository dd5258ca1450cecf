"""The graph primitives of csrc/prims.cu compared exactly, on every path they choose: the exclusive scan
(dm_scan_exclusive_u32), the LSD radix sort (dm_sort_edges), the hashed run reduction (dm_edges_sort_unique,
dm_rag_finish, dm_rag_build) and the bucket sort (dm_csr_build by the low key half with CSR offsets, dm_merge_apply by
the high half without values), each against a numpy restatement of its header text: np.unique, a stable argsort,
sums mod 2^32 and a uint32 cumsum.

Which path a sort takes depends only on its input, so a case could miss the path it is meant to cover and still pass.
Every GPU case therefore asserts its path twice:
  * the rule: a numpy restatement of the choice in prims.cu (unique_rule, bucket_rule below);
  * the probe: what the kernel did, read back from its workspace.  The last piece of carve_ws is `misc`, 16 words in a
    256-byte piece of their own; launch_coop zeroes words 0 and 1 before the hashed and the bucket kernels.  Word 0
    counts the buckets with HUB_MIN < size <= hub limit (it keeps counting past HUB_CAP), word 1 is the fall-back flag.
    The sort workspace is the last piece of the layouts of dm_edges_sort_unique, dm_rag_finish and dm_csr_build, so
    misc sits at ws + query - 256; dm_merge_apply keeps one int64 behind it, so there it is at ws + query - 512.  The
    workspace starts filled with a sentinel: the radix sort never touches misc, so the host's choice of the radix sort
    shows as an untouched sentinel.
The CPU tests check these layout facts and the thresholds against the sources, so that a layout change fails here
instead of making the probe read noise.  The test ids name the path: hashed, hashed-hubs, bucket, bucket-hubs,
fb-hubsize, fb-hubcount, fb-range (the radix sort taken inside the launch), host-radix, radix-pN (N passes).

Every output buffer sits between guard bytes, garbage behind the count must be ignored and left as it was, and every
call is made twice with bit-equal results.
"""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "deepmerge_b200", "csrc")

U64 = np.uint64
SENT = 0xFFFFFFFFFFFFFFFF                   # ~0: the default sentinel of the run reduction
WS_FILL = 0xA7                              # workspace sentinel
WS_WORD = 0xA7A7A7A7
GUARD, FILL = 4096, 0xA5                    # guard bytes on each side of an output, and their value

# thresholds of prims.cu (checked against the source by test_thresholds_match_the_source)
HUB_MIN, HUB_MAX, HUB_CAP, HUB_MAX_SORT = 48, 4096, 1024, 2048
SORT_TILE = SCAN_TILE = 2048
HASH_MAX_GRID = 1024
# blocks per SM of the hashed and bucket kernels: the cap passed to coop_grid_limit, which is also their
# __launch_bounds__ minimum.  That 4 blocks of these kernels really fit on an SM is not measured; the sweep cases below
# assume it.
BLOCKS_PER_SM = 4
HB = 4                                      # items per thread and step in the hashed / bucket kernels


def src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


# ------------------------------------------------------------------------------------------
# path rules (prims.cu: sort_unique / sort_pairs on the host, edge_unique_hashed / bucket_sort_fused in the launch)
# ------------------------------------------------------------------------------------------
def bits_for(n):
    b = 1
    while b < 32 and (1 << b) < n:
        b += 1
    return b


def radix_passes(n_regions):
    return -(-2 * bits_for(n_regions) // 9)


def choose(range_bad, deg, hub_max, small, hubs_name):
    """-> (path, (hub count, fall-back flag)) from the bucket sizes `deg` and whether an id was out of range."""
    deg = np.asarray(deg, np.int64)
    hubs = int(((deg > HUB_MIN) & (deg <= hub_max)).sum())
    big = bool((deg > hub_max).any())
    if range_bad:
        path = "fb-range"
    elif big:
        path = "fb-hubsize"
    elif hubs > HUB_CAP:
        path = "fb-hubcount"
    else:
        path = hubs_name if hubs else small
    return path, (hubs, int(range_bad or big or hubs > HUB_CAP))


def unique_rule(keys, n_ids, cap, sentinel=SENT):
    """sort_unique: the radix sort chosen on the host (misc untouched: None), or the hashed kernel and what it leaves in
    misc.  keys are the n pairs it reads."""
    if not (0 < n_ids <= 4 * cap + 65536 and cap < 2 ** 31):
        return "host-radix", None
    k = np.asarray(keys, U64)
    k = k[k != U64(sentinel)]
    bad = ((k >> U64(32)) >= U64(n_ids)) | (k == U64(SENT))
    u = np.unique(k[~bad])
    deg = np.bincount((u >> U64(32)).astype(np.int64), minlength=n_ids)
    return choose(bool(bad.any()), deg, HUB_MAX, "hashed", "hashed-hubs")


def bucket_rule(primary, n_ids):
    """bucket_sort_fused: raw pairs per primary id, HUB_MAX_SORT as the hub limit, no host branch."""
    p = np.asarray(primary, np.int64)
    bad = p >= n_ids
    deg = np.bincount(p[~bad], minlength=n_ids)
    return choose(bool(bad.any()), deg, HUB_MAX_SORT, "bucket", "bucket-hubs")


# ------------------------------------------------------------------------------------------
# restatements of the header text
# ------------------------------------------------------------------------------------------
def pack(lo, hi):
    return (np.asarray(lo, U64) << U64(32)) | np.asarray(hi, U64)


def unique_ref(keys, lens, sentinel=SENT):
    """Unique keys ascending (sentinel dropped) and their lengths summed mod 2^32."""
    keep = keys != U64(sentinel)
    uk, inv = np.unique(keys[keep], return_inverse=True)
    s = np.zeros(uk.shape[0], U64)
    np.add.at(s, inv, lens[keep].astype(U64))
    return uk, (s & U64(0xFFFFFFFF)).astype(np.uint32)


def scan_ref(x):
    c = np.cumsum(x.astype(U64), dtype=U64)          # wraps mod 2^64, so mod 2^32 stays exact
    ex = np.concatenate([[U64(0)], c[:-1]]) if x.size else c
    return (ex & U64(0xFFFFFFFF)).astype(np.uint32), int(c[-1] & U64(0xFFFFFFFF)) if x.size else 0


# ------------------------------------------------------------------------------------------
# CPU: the rules on hand-built degree vectors, and the layout facts the probe relies on
# ------------------------------------------------------------------------------------------
def test_thresholds_match_the_source():
    s = src("prims.cu")
    h = src("prims.cuh")

    def const(name, text=s):
        m = re.search(r"\b%s\s*=\s*(\d+)\b" % name, text)
        assert m, name
        return int(m.group(1))
    assert (const("HUB_MIN"), const("HUB_MAX"), const("HUB_CAP")) == (HUB_MIN, HUB_MAX, HUB_CAP)
    assert const("HUB_MAX_SORT") == HUB_MAX_SORT
    assert const("HASH_MAX_GRID") == HASH_MAX_GRID and const("HASH_BLOCKS_PER_SM") == BLOCKS_PER_SM
    assert const("HB") == HB
    assert const("SORT_THREADS", h) * const("SORT_ITEMS", h) == SORT_TILE
    assert const("SCAN_THREADS", h) * const("SCAN_ITEMS", h) == SCAN_TILE
    # grids: radix min(tiles, 2 per SM); hashed and bucket at most HASH_BLOCKS_PER_SM per SM and HASH_MAX_GRID, the
    # bucket sort also at most 5 S / 2; the per-SM cap is the __launch_bounds__ minimum of both kernels
    assert "imin64(ceil_div(cap, SORT_TILE), coop_grid_limit((const void*)radix_sort_fused, 2))" in s
    assert "imin64(coop_grid_limit((const void*)edge_unique_hashed, HASH_BLOCKS_PER_SM), HASH_MAX_GRID)" in s
    assert "imin64(ceil_div(imax64(cap, n_ids), SORT_THREADS * 4), limit)" in s
    assert "imin64(coop_grid_limit((const void*)bucket_sort_fused, HASH_BLOCKS_PER_SM), HASH_MAX_GRID)" in s
    assert "imin64(imin64(ceil_div(imax64(cap, n_ids), SORT_THREADS), limit), 5 * num_sms() / 2)" in s
    assert len(re.findall(r"__launch_bounds__\(SORT_THREADS, HASH_BLOCKS_PER_SM\)", s)) == 2
    # the host's choice of sort_unique
    assert "int64_t hash_ids_cap(int64_t cap) { return 4 * cap + 65536; }" in s
    assert "if (!(n_ids > 0 && n_ids <= hash_ids_cap(cap) && key_bits == 2 * id_bits && cap < (1ll << 31)))" in s
    # the in-launch rules: sizes above HUB_MIN are hubs up to the limit, counted in misc[0]; the flag is misc[1]
    assert "bucket_offsets_phase(H, sm, shift, HUB_MAX);" in s
    assert "bucket_offsets_phase(H, sm, shift, HUB_MAX_SORT);" in s
    body = s[s.index("void bucket_offsets_phase"):s.index("bucket_chunk_bases")]
    for frag in ("if (d > HUB_MIN) {", "if (d > hub_max) {", "atomicAdd(H.misc, 1u)", "if (slot < HUB_CAP)",
                 "atomicExch(H.misc + 1, 1u)"):
        assert frag in body, frag
    assert "if (pend[u] && ((int64_t)lo >= H.n_ids || key[u] == ~0ull)) {" in s
    assert "if ((int64_t)p >= H.n_ids) atomicExch(H.misc + 1, 1u);" in s


def test_misc_is_the_last_piece_of_every_probed_layout():
    s = src("prims.cu")
    carve = s[s.index("size_t carve_ws("):]
    carve = carve[:carve.index("\n}\n")]
    takes = re.findall(r"c\.take<[^>]+>\([^;]*\);", carve)
    assert takes[-1] == "c.take<unsigned>(16);" and "H.misc = c.take<unsigned>(16);" in carve
    assert carve.rstrip().endswith("return c.used();")
    assert "unsigned* misc;" in s and "if (misc) DM_CUDA(cudaMemsetAsync(misc, 0, 4 * sizeof(unsigned), s));" in s
    com = src("common.cuh")
    assert "off = align_up(off, 256);" in com and "size_t used() const { return align_up(off, 256); }" in com
    # the sort workspace ends the layouts of dm_rag_finish, dm_edges_sort_unique and dm_csr_build ...
    rag = src("rag.cu")
    assert ("return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<char>(prims::ws_bytes(cap, true)), "
            "c.used()};") in rag
    assert ("return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<int64_t>(1), "
            "c.take<char>(prims::ws_bytes(cap, true)),\n            c.used()};") in rag
    assert ("return {c.take<uint64_t>(cap), c.take<uint32_t>(cap), c.take<int64_t>(1),\n"
            "            c.take<char>(prims::ws_bytes(cap, false, n_regions + 1)), c.used()};") in src("pool.cu")
    # ... and dm_merge_apply's list comes first, the sort workspace and one int64 (the list length) after it
    assert ("return {c.take<uint64_t>(cap), c.take<char>(prims::ws_bytes(cap, false)), c.take<int64_t>(1), "
            "c.used()};") in src("merge.cu")


def test_rules_at_every_threshold():
    d = np.zeros(100, np.int64)
    assert choose(False, d, HUB_MAX, "hashed", "hashed-hubs") == ("hashed", (0, 0))
    d[7] = HUB_MIN
    assert choose(False, d, HUB_MAX, "hashed", "hashed-hubs") == ("hashed", (0, 0))
    d[7] = HUB_MIN + 1
    assert choose(False, d, HUB_MAX, "hashed", "hashed-hubs") == ("hashed-hubs", (1, 0))
    d[7] = HUB_MAX
    assert choose(False, d, HUB_MAX, "hashed", "hashed-hubs") == ("hashed-hubs", (1, 0))
    d[7] = HUB_MAX + 1
    assert choose(False, d, HUB_MAX, "hashed", "hashed-hubs") == ("fb-hubsize", (0, 1))
    assert choose(False, d, HUB_MAX_SORT, "bucket", "bucket-hubs") == ("fb-hubsize", (0, 1))
    d[7] = HUB_MAX_SORT
    assert choose(False, d, HUB_MAX_SORT, "bucket", "bucket-hubs") == ("bucket-hubs", (1, 0))
    d[7] = HUB_MAX_SORT + 1
    assert choose(False, d, HUB_MAX_SORT, "bucket", "bucket-hubs") == ("fb-hubsize", (0, 1))
    h = np.full(HUB_CAP, HUB_MIN + 1)
    assert choose(False, h, HUB_MAX, "hashed", "hashed-hubs") == ("hashed-hubs", (HUB_CAP, 0))
    h = np.full(HUB_CAP + 1, HUB_MIN + 1)
    assert choose(False, h, HUB_MAX, "hashed", "hashed-hubs") == ("fb-hubcount", (HUB_CAP + 1, 1))
    assert choose(True, np.ones(5), HUB_MAX, "hashed", "hashed-hubs") == ("fb-range", (0, 1))
    # the host's choice
    k = pack([0, 1], [1, 2])
    assert unique_rule(k, 4 * 1000 + 65536, 1000)[0] == "hashed"
    assert unique_rule(k, 4 * 1000 + 65537, 1000) == ("host-radix", None)
    assert unique_rule(k, 0, 1000) == ("host-radix", None)
    # the range rule looks at the first id only; ~0 is the sentinel, not an out-of-range key
    assert unique_rule(pack([9, 0], [0, 9]), 10, 100)[0] == "hashed"
    assert unique_rule(pack([10, 0], [0, 9]), 10, 100)[0] == "fb-range"
    assert unique_rule(np.array([SENT, 5], U64), 10, 100)[0] == "hashed"
    assert unique_rule(np.array([SENT, 5], U64), 10, 100, sentinel=pack(10, 10))[0] == "fb-range"
    # unique keys count, not raw pairs
    assert unique_rule(np.repeat(pack(np.zeros(49), np.arange(49)), 3), 100, 1000)[1] == (1, 0)
    assert unique_rule(np.repeat(pack(np.zeros(48), np.arange(48)), 3), 100, 1000)[1] == (0, 0)
    assert bucket_rule(np.r_[np.zeros(HUB_MIN), 1], 3) == ("bucket", (0, 0))
    assert bucket_rule(np.r_[np.zeros(HUB_MIN + 1), 1], 3) == ("bucket-hubs", (1, 0))
    assert bucket_rule([0, 3], 3) == ("fb-range", (0, 1))
    assert [radix_passes(r) for r in (1, 16, 17, 512, 513, 8192, 8193, 1 << 18, (1 << 18) + 1, 1 << 22, 1 << 27,
                                      2 ** 31 - 1, 2 ** 31, 2 ** 32)] == [1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 7, 7, 8]


def test_restatements():
    k = np.array([5, SENT, 3, 5, 3, 3], U64)
    ln = np.array([2 ** 32 - 1, 7, 1, 2, 2, 3], np.uint32)
    uk, s = unique_ref(k, ln)
    assert uk.tolist() == [3, 5] and s.tolist() == [6, 1]
    ex, tot = scan_ref(np.array([2 ** 32 - 1, 2, 3], np.uint32))
    assert ex.tolist() == [0, 2 ** 32 - 1, 1] and tot == 4
    assert scan_ref(np.zeros(0, np.uint32))[1] == 0


# ------------------------------------------------------------------------------------------
# device helpers
# ------------------------------------------------------------------------------------------
def lib():
    from deepmerge_b200._lib import lib as _l
    return _l()


def sms():
    n = lib().dm_num_sms()
    assert n > 0
    return n


def hashed_sweep(S):
    """Pairs that one step of the hashed kernel's insert loop covers when its grid is at its limit."""
    return HB * 256 * min(BLOCKS_PER_SM * S, HASH_MAX_GRID)


def radix_sweep(S):
    """Pairs the radix sort's tile loop covers in one step at its grid limit of 2 blocks per SM."""
    return SORT_TILE * 2 * S


def bucket_sweep(S):
    return HB * 256 * min(BLOCKS_PER_SM * S, HASH_MAX_GRID, 5 * S // 2)


class Guarded:
    """nbytes of device memory with `guard` bytes of FILL on each side; the region starts as `init` (or FILL)."""

    def __init__(self, nbytes, init=None, guard=GUARD):
        import torch
        self.n, self.g = int(nbytes), guard
        self.buf = torch.full((2 * guard + self.n,), FILL, dtype=torch.uint8, device="cuda")
        self.t = self.buf[guard:guard + self.n]
        if init is not None:
            b = np.ascontiguousarray(init).view(np.uint8).reshape(-1)
            assert b.shape[0] == self.n
            self.t.copy_(torch.from_numpy(b).cuda())

    def ptr(self):
        return self.t.data_ptr()

    def get(self, dtype):
        return self.t.cpu().numpy().view(dtype)

    def intact(self):
        b = self.buf.cpu().numpy()
        return bool((b[:self.g] == FILL).all() and (b[self.g + self.n:] == FILL).all())


def workspace(nbytes):
    import torch
    return torch.full((int(nbytes),), WS_FILL, dtype=torch.uint8, device="cuda")


def probe(ws, off):
    return tuple(int(x) for x in ws[off:off + 8].cpu().numpy().view(np.uint32))


def check_probe(ws, off, misc):
    """misc None: the radix sort chosen on the host left both words as they were."""
    got = probe(ws, off)
    assert got == ((WS_WORD, WS_WORD) if misc is None else misc), "probe %s, rule %s" % (got, misc)


def sync():
    import torch
    torch.cuda.synchronize()


def garbage_keys(rng, m, R):
    """Keys a wrong count would pick up: ~0, ids far out of range, and ordinary keys."""
    g = pack(rng.integers(0, 1 << 31, m), rng.integers(0, 1 << 31, m))
    g[::3] = U64(SENT)
    g[1::3] = pack(rng.integers(0, R, m), rng.integers(0, R, m))[1::3]
    return g


# ------------------------------------------------------------------------------------------
# run reduction: dm_edges_sort_unique
# ------------------------------------------------------------------------------------------
def gen_random(rng, n, R):
    return pack(rng.integers(0, R, n), rng.integers(0, R, n))


def gen_bucket(size, R, fill_deg=8):
    """One first id (5) with `size` distinct partners, each listed twice; every other first id below R has a few."""
    def g(rng, n, _R):
        hub = np.repeat(pack(np.full(size, 5), rng.permutation(R)[:size]), 2)
        rest = pack(rng.integers(0, R, n - hub.size), rng.integers(0, fill_deg, n - hub.size))
        rest[(rest >> U64(32)) == U64(5)] = pack(6, 0)
        k = np.concatenate([hub, rest])
        return k[rng.permutation(k.size)]
    return g


def gen_hubs(count, size=HUB_MIN + 1):
    """`count` first ids with `size` distinct partners each (each listed twice), then small buckets."""
    def g(rng, n, R):
        lo = np.repeat(np.arange(count), size)
        hi = np.tile(np.arange(size), count)
        k = np.repeat(pack(lo, hi), 2)
        rest = pack(rng.integers(count, R, n - k.size), rng.integers(0, 8, n - k.size))
        k = np.concatenate([k, rest])
        return k[rng.permutation(k.size)]
    return g


def gen_first(first):
    def g(rng, n, R):
        k = gen_random(rng, n, R)
        k[rng.choice(n, 5, replace=False)] = pack(first, rng.integers(0, R, 5))
        return k
    return g


def gen_equal(rng, n, R):
    return np.full(n, pack(R - 1, R // 2), U64)


def gen_ascending(rng, n, R):
    v = np.sort(rng.choice(R * R, n, replace=False))
    return pack(v // R, v % R)


def gen_descending(rng, n, R):
    return gen_ascending(rng, n, R)[::-1].copy()


def gen_far_dups(rng, n, R):
    """1000 distinct keys repeated all over: every run crosses tiles and blocks."""
    base = gen_random(rng, 1000, R)
    return base[rng.integers(0, 1000, n)]


def gen_top(R):
    """Keys whose ids include 2^b - 1 for n_regions = 2^b or 2^b + 1."""
    def g(rng, n, _R):
        top = (1 << (bits_for(R) if R & (R - 1) == 0 else bits_for(R) - 1)) - 1
        k = gen_random(rng, n, top + 1)
        k[:20] = pack(top, rng.integers(0, top + 1, 20))
        k[20:40] = pack(rng.integers(0, top + 1, 20), top)
        return k
    return g


def with_sentinels(g):
    """n // 10 entries of ~0 inserted among the keys of g."""
    def h(rng, n, R):
        k = g(rng, n - n // 10, R)
        return np.insert(k, rng.integers(0, k.size + 1, n // 10), U64(SENT))
    return h


HOST = lambda cap: 4 * cap + 65537           # smallest n_regions for which the host chooses the radix sort

# (path, generator, n, n_regions, extra capacity, n_dev: None = n, lens: "small" / "wrap")
UNIQUE_CASES = [
    ("hashed", "random", gen_random, 20000, 1000, 33, None, "small"),
    ("hashed-hubs", "random", gen_random, 20000, 100, 33, None, "small"),
    ("hashed", "bucket48", gen_bucket(HUB_MIN, 5000), 20000, 5000, 33, None, "small"),
    ("hashed-hubs", "bucket49", gen_bucket(HUB_MIN + 1, 5000), 20000, 5000, 33, None, "small"),
    ("hashed-hubs", "bucket4096", gen_bucket(HUB_MAX, 5000), 30000, 5000, 33, None, "small"),
    ("fb-hubsize", "bucket4097", gen_bucket(HUB_MAX + 1, 5000), 30000, 5000, 33, None, "small"),
    ("hashed-hubs", "hubs1024", gen_hubs(HUB_CAP), 110000, 1100, 33, None, "small"),
    ("fb-hubcount", "hubs1025", gen_hubs(HUB_CAP + 1), 110000, 1100, 33, None, "small"),
    ("hashed", "first-nids-1", gen_first(999), 20000, 1000, 33, None, "small"),
    ("fb-range", "first-nids", gen_first(1000), 20000, 1000, 33, None, "small"),
    ("fb-range", "first-top", gen_first(1023), 20000, 1000, 33, None, "small"),
    ("hashed", "host-limit", gen_random, 900, "4cap+65536", 100, None, "small"),
    ("host-radix", "host-limit+1", gen_random, 900, "4cap+65537", 100, None, "small"),
    ("hashed", "all-equal-wrap", gen_equal, 100000, 1000, 33, None, "wrap"),
    ("host-radix", "all-equal-wrap", gen_equal, 100000, 1 << 20, 33, None, "wrap"),
    ("hashed", "distinct-ascending", gen_ascending, 50000, 5000, 33, None, "small"),
    ("hashed", "distinct-descending", gen_descending, 50000, 5000, 33, None, "small"),
    ("host-radix", "distinct-descending", gen_descending, 50000, 1 << 20, 33, None, "small"),
    ("hashed", "far-dups-wrap", gen_far_dups, 3000000, 1000, 777, None, "wrap"),
    ("host-radix", "far-dups-wrap", gen_far_dups, 3000000, 1 << 24, 777, None, "wrap"),
    ("hashed", "top-2^12", gen_top(4096), 50000, 4096, 33, None, "small"),
    ("hashed", "top-2^12+1", gen_top(4097), 50000, 4097, 33, None, "small"),
    ("host-radix", "top-2^20", gen_top(1 << 20), 50000, 1 << 20, 33, None, "small"),
    ("hashed", "sentinels", with_sentinels(gen_random), 20000, 1000, 33, None, "small"),
    ("hashed-hubs", "sentinels", with_sentinels(gen_random), 20000, 100, 33, None, "small"),
    ("fb-hubsize", "sentinels", with_sentinels(gen_bucket(HUB_MAX + 1, 5000)), 30000, 5000, 33, None, "small"),
    ("fb-hubcount", "sentinels", with_sentinels(gen_hubs(HUB_CAP + 1)), 125000, 1100, 33, None, "small"),
    ("fb-range", "sentinels", with_sentinels(gen_first(1000)), 20000, 1000, 33, None, "small"),
    ("host-radix", "sentinels", with_sentinels(gen_random), 20000, 1 << 20, 33, None, "small"),
    ("hashed", "n0", gen_random, 0, 1000, 500, None, "small"),
    ("host-radix", "n0", gen_random, 0, 1 << 20, 500, None, "small"),
    ("hashed", "over-cap", gen_random, 5000, 1000, 0, 5000 + 2047, "small"),
    ("fb-range", "over-cap", gen_first(1000), 5000, 1000, 0, 1 << 40, "small"),
    ("host-radix", "over-cap", gen_random, 5000, 1 << 20, 0, 5001, "small"),
    ("hashed", "n2047", gen_random, 2047, 1000, 1, None, "small"),
    ("hashed", "n2048", gen_random, 2048, 1000, 1, None, "small"),
    ("hashed", "n2049", gen_random, 2049, 1000, 1, None, "small"),
    ("host-radix", "n2047", gen_random, 2047, 1 << 20, 1, None, "small"),
    ("host-radix", "n2048", gen_random, 2048, 1 << 20, 1, None, "small"),
    ("host-radix", "n2049", gen_random, 2049, 1 << 20, 1, None, "small"),
    ("hashed", "sweep", gen_random, "hashed+0", 100000, 100, None, "small"),
    ("hashed", "sweep+1", gen_random, "hashed+1", 100000, 100, None, "small"),
    ("host-radix", "sweep", gen_random, "radix+0", 1 << 24, 100, None, "small"),
    ("host-radix", "sweep+1", gen_random, "radix+1", 1 << 24, 100, None, "small"),
    ("hashed", "3M", gen_random, 3000000, 1 << 20, 5, None, "small"),
    ("fb-hubcount", "3M", gen_random, 3000000, 2500, 5, None, "small"),
]


def resolve_n(n, S):
    if isinstance(n, str):
        kind, d = n.split("+")
        return {"hashed": hashed_sweep, "radix": radix_sweep, "bucket": bucket_sweep}[kind](S) + int(d)
    return n


def unique_case_params():
    out = []
    for path, name, gen, n, R, extra, ndev, lens in UNIQUE_CASES:
        for alias in ((False, True) if name in ("random", "bucket4097", "hubs1025", "first-nids", "host-limit+1",
                                                "over-cap") else (False,)):
            out.append(pytest.param(path, gen, n, R, extra, ndev, lens, alias,
                                    id="%s-%s%s" % (path, name, "-alias" if alias else "")))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("path,gen,n,R,extra,ndev,lens,alias", unique_case_params())
def test_edges_sort_unique_exact(cuda, path, gen, n, R, extra, ndev, lens, alias):
    """dm_edges_sort_unique: keys[0, E) / lens[0, E) are the unique keys of the n = min(*n_in, capacity) pairs with
    their lengths summed mod 2^32, ~0 dropped; *n_out = E (n_out may be n_in); keys and lens from n on are not
    touched."""
    L = lib()
    S = sms()
    n = resolve_n(n, S)
    cap = n + extra
    if isinstance(R, str):
        R = {"4cap+65536": 4 * cap + 65536, "4cap+65537": HOST(cap)}[R]
    rng = np.random.default_rng(n + R + extra)
    keys = np.concatenate([gen(rng, n, R) if n else np.zeros(0, U64), garbage_keys(rng, extra, R)])
    if lens == "wrap":
        ln = rng.integers(1 << 30, 1 << 32, cap, dtype=np.uint64).astype(np.uint32)
    else:
        ln = rng.integers(1, 1000, cap).astype(np.uint32)
    n_dev = n if ndev is None else ndev
    m = min(n_dev, cap)
    rule, misc = unique_rule(keys[:m], R, cap)
    assert rule == path
    uk, us = unique_ref(keys[:m], ln[:m])
    query = L.dm_edges_unique_workspace_bytes(cap)
    results = []
    for _ in range(2):
        k, v = Guarded(cap * 8, keys), Guarded(cap * 4, ln)
        nin = Guarded(8, np.array([n_dev], np.int64))
        nout = nin if alias else Guarded(8, np.array([-7], np.int64))
        ws = workspace(query)
        L.check(L.dm_edges_sort_unique(k.ptr(), v.ptr(), nin.ptr(), cap, R, nout.ptr(), ws.data_ptr(), query, None),
                "dm_edges_sort_unique")
        sync()
        check_probe(ws, query - 256, misc)
        gk, gv, E = k.get(U64), v.get(np.uint32), int(nout.get(np.int64)[0])
        assert E == uk.shape[0]
        assert np.array_equal(gk[:E], uk)
        assert np.array_equal(gv[:E], us)
        assert np.array_equal(gk[m:], keys[m:]) and np.array_equal(gv[m:], ln[m:]), "the tail behind n changed"
        if not alias:
            assert int(nin.get(np.int64)[0]) == n_dev
        assert k.intact() and v.intact() and nin.intact() and nout.intact()
        results.append((gk[:E].copy(), gv[:E].copy()))
    assert all(np.array_equal(a, b) for a, b in zip(*results))


# ------------------------------------------------------------------------------------------
# run reduction: dm_rag_finish on a raw list placed in its workspace, and dm_rag_build through the radix sort
# ------------------------------------------------------------------------------------------
def rag_raw_offsets(cap):
    """rag.cu rag_ws: raw keys, raw counts, then the sort workspace (256-byte aligned pieces)."""
    a = -(-cap * 8 // 256) * 256
    return 0, a


RAG_CASES = [
    ("hashed", "random", gen_random, 20000, 1000, 100, None),
    ("hashed-hubs", "random", gen_random, 20000, 100, 100, None),
    ("fb-hubsize", "bucket4097", gen_bucket(HUB_MAX + 1, 5000), 30000, 5000, 100, None),
    ("fb-hubcount", "hubs1025", gen_hubs(HUB_CAP + 1), 110000, 1100, 100, None),
    ("fb-range", "first-nids", gen_first(1000), 20000, 1000, 100, None),
    ("host-radix", "host-limit+1", gen_random, 20000, "4cap+65537", 100, None),
    ("hashed", "counts1-over-cap", gen_random, 20000, 1000, 0, 20000 + 12345),
    ("host-radix", "counts1-over-cap", gen_random, 20000, 1 << 20, 0, 20000 + 12345),
    ("hashed", "n0", gen_random, 0, 1000, 64, None),
]


@pytest.mark.gpu
@pytest.mark.parametrize("path,gen,n,R,extra,c1", [pytest.param(*c[:1], *c[2:], id="%s-%s" % c[:2]) for c in RAG_CASES])
def test_rag_finish_exact(cuda, path, gen, n, R, extra, c1):
    """dm_rag_finish reduces min(counts[1], capacity) raw entries: ascending unique edge_keys, boundary_len summed,
    counts[0] = E; counts[1..3] stay as they were."""
    import torch
    L = lib()
    cap = n + extra
    if isinstance(R, str):
        R = HOST(cap)
    rng = np.random.default_rng(3 * n + R)
    raw = np.concatenate([gen(rng, n, R) if n else np.zeros(0, U64), garbage_keys(rng, extra, R)])
    cnt = rng.integers(1, 1 << 20, cap).astype(np.uint32)
    c1 = n if c1 is None else c1
    m = min(c1, cap)
    rule, misc = unique_rule(raw[:m], R, cap)
    assert rule == path
    uk, us = unique_ref(raw[:m], cnt[:m])
    query = L.dm_rag_workspace_bytes(cap)
    ok, oc = rag_raw_offsets(cap)
    prev = None
    for _ in range(2):
        ws = workspace(query)
        ws[ok:ok + cap * 8].copy_(torch.from_numpy(raw.view(np.uint8)).cuda())
        ws[oc:oc + cap * 4].copy_(torch.from_numpy(cnt.view(np.uint8)).cuda())
        ek0 = rng.integers(0, 1 << 62, cap).astype(U64)
        bl0 = rng.integers(0, 1 << 31, cap).astype(np.uint32)
        ek, bl = Guarded(cap * 8, ek0), Guarded(cap * 4, bl0)
        counts0 = np.array([-1, c1, 3, 4], np.int64)
        counts = Guarded(32, counts0)
        L.check(L.dm_rag_finish(ek.ptr(), bl.ptr(), cap, R, counts.ptr(), ws.data_ptr(), query, None), "dm_rag_finish")
        sync()
        check_probe(ws, query - 256, misc)
        got_c = counts.get(np.int64)
        E = int(got_c[0])
        assert E == uk.shape[0] and np.array_equal(got_c[1:], counts0[1:])
        gk, gb = ek.get(U64), bl.get(np.uint32)
        assert np.array_equal(gk[:E], uk) and np.array_equal(gb[:E], us)
        assert np.array_equal(gk[E:], ek0[E:]) and np.array_equal(gb[m:], bl0[m:])
        assert ek.intact() and bl.intact() and counts.intact()
        if prev is not None:
            assert np.array_equal(prev[0], gk[:E]) and np.array_equal(prev[1], gb[:E])
        prev = (gk[:E].copy(), gb[:E].copy())


@pytest.mark.gpu
def test_rag_build_through_the_radix_sort_with_an_odd_pass_count(cuda):
    """host-radix-p5: labels are a sparse subset of [0, 2^20 + 1) (21-bit ids, 42-bit keys: 5 radix passes) and the
    capacity is small enough that n_regions > 4 capacity + 65536, so the run reduction follows an odd number of passes."""
    from oracle import oracle_np as o
    L = lib()
    R = (1 << 20) + 1
    assert radix_passes(R) == 5
    rng = np.random.default_rng(11)
    ids = np.r_[rng.choice(R - 1, 300, replace=False), R - 1, 0].astype(np.int32)
    small = ids[rng.integers(0, ids.size, (24, 40))]
    lab = np.kron(small, np.ones((3, 4), np.int32))
    lab[rng.random(lab.shape) < 0.05] = R - 1
    H, W = lab.shape
    cap = 40000
    assert R > 4 * cap + 65536
    keys, blen, area, _ = o.build_rag(lab, R)
    query = L.dm_rag_workspace_bytes(cap)
    import torch
    lab_d = torch.from_numpy(lab).cuda()
    a = torch.zeros(R, dtype=torch.int64, device="cuda")
    b = torch.zeros(R, dtype=torch.int64, device="cuda")
    ek, bl = Guarded(cap * 8), Guarded(cap * 4)
    counts = Guarded(32)
    ws = workspace(query)
    L.check(L.dm_rag_build(lab_d.data_ptr(), H, H, W, W, None, 0, 0, R, 1, 1, a.data_ptr(), b.data_ptr(), None, None,
                           ek.ptr(), bl.ptr(), cap, counts.ptr(), ws.data_ptr(), query, None), "dm_rag_build")
    sync()
    check_probe(ws, query - 256, None)
    c = counts.get(np.int64)
    assert c[2] == 0 and c[0] == keys.shape[0]
    assert np.array_equal(ek.get(U64)[:c[0]], keys) and np.array_equal(bl.get(np.uint32)[:c[0]], blen)
    assert np.array_equal(a.cpu().numpy(), area)
    assert ek.intact() and bl.intact() and counts.intact()


# ------------------------------------------------------------------------------------------
# radix sort: dm_sort_edges (the radix sort always: it passes no id count)
# ------------------------------------------------------------------------------------------
SORT_CASES = [(r, n) for r in (1, 512, 8192, 1 << 18, 1 << 22, 1 << 27, 2 ** 31 - 1, 2 ** 32) for n in (5000,)] + [
    (1, 100000), (3, 300000), (70000, 2047), (70000, 2048), (70000, 2049), (70000, "radix+0"), (70000, "radix+1"),
    (1 << 22, 3000000)]


def sort_params():
    out = []
    for R, n in SORT_CASES:
        for vals in (True, False):
            out.append(pytest.param(R, n, vals, None, id="radix-p%d-R%d-n%s-%s" % (radix_passes(R), R, n,
                                                                                    "vals" if vals else "novals")))
    for ndev in (0, "over"):
        out.append(pytest.param(1000, 3000, True, ndev, id="radix-p%d-ndev-%s" % (radix_passes(1000), ndev)))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("R,n,vals,ndev", sort_params())
def test_sort_edges_exact(cuda, R, n, vals, ndev):
    """dm_sort_edges: a stable sort of the n = min(*n_dev, capacity) pairs by key, values with them (vals nullable);
    the pairs from n on are not touched.  Every pass count from 1 to 8, odd ones ending in the copy back home; R = 1 and
    3 give long runs of equal keys with distinct values."""
    L = lib()
    n = resolve_n(n, sms())
    extra = 0 if ndev == "over" else 123
    cap = n + extra
    n_dev = {None: n, 0: 0, "over": n + 5000}[ndev]
    m = min(n_dev, cap)
    rng = np.random.default_rng(n + R % 1000003)
    keys = np.concatenate([pack(rng.integers(0, R, n), rng.integers(0, R, n)), garbage_keys(rng, extra, R)])
    v0 = rng.permutation(cap).astype(np.uint32)
    order = np.argsort(keys[:m], kind="stable")
    query = L.dm_sort_edges_workspace_bytes(cap)
    prev = None
    for _ in range(2):
        k = Guarded(cap * 8, keys)
        v = Guarded(cap * 4, v0) if vals else None
        nd = Guarded(8, np.array([n_dev], np.int64))
        ws = workspace(query)
        L.check(L.dm_sort_edges(k.ptr(), v.ptr() if vals else None, nd.ptr(), cap, R, ws.data_ptr(), query, None),
                "dm_sort_edges")
        sync()
        check_probe(ws, query - 256, None)
        gk = k.get(U64)
        assert np.array_equal(gk[:m], keys[:m][order]) and np.array_equal(gk[m:], keys[m:])
        assert k.intact() and nd.intact()
        if vals:
            gv = v.get(np.uint32)
            assert np.array_equal(gv[:m], v0[:m][order]) and np.array_equal(gv[m:], v0[m:])
            assert v.intact()
            gk = np.concatenate([gk.view(np.uint8), gv.view(np.uint8)])
        if prev is not None:
            assert np.array_equal(prev, gk)
        prev = gk.copy()


# ------------------------------------------------------------------------------------------
# bucket sort: dm_csr_build (by the low half, CSR offsets) and dm_merge_apply (by the high half, no values)
# ------------------------------------------------------------------------------------------
def rop_random(rng, N, R):
    return rng.integers(-1, R + 2, N).astype(np.int32)    # -1, R and R + 1 have no region


def rop_region(size, count=1):
    """`count` regions of `size` points each, the rest spread over the other regions."""
    def g(rng, N, R):
        r = rng.integers(count, R, N).astype(np.int32)
        pick = rng.choice(N, size * count, replace=False)
        r[pick] = np.repeat(np.arange(count), size)
        return r
    return g


def rop_invalid(k):
    def g(rng, N, R):
        r = rng.integers(0, R, N).astype(np.int32)
        r[rng.choice(N, k, replace=False)] = -1
        return r
    return g


CSR_CASES = [
    ("bucket", "random", rop_random, 3000, 500),
    ("bucket", "regions-over-points", rop_random, 1000, 200000),
    ("bucket", "region48", rop_region(HUB_MIN), 20000, 5000),
    ("bucket-hubs", "region49", rop_region(HUB_MIN + 1), 20000, 5000),
    ("bucket-hubs", "region2048", rop_region(HUB_MAX_SORT), 20000, 5000),
    ("fb-hubsize", "region2049", rop_region(HUB_MAX_SORT + 1), 20000, 5000),
    ("bucket-hubs", "regions1024x49", rop_region(HUB_MIN + 1, HUB_CAP), 60000, 20000),
    ("fb-hubcount", "regions1025x49", rop_region(HUB_MIN + 1, HUB_CAP + 1), 60000, 20000),
    ("bucket-hubs", "invalid2048", rop_invalid(2048), 20000, 15000),
    ("fb-hubsize", "invalid2049", rop_invalid(2049), 20000, 15000),
    ("bucket", "n2047", rop_random, 2047, 5000),
    ("bucket", "n2048", rop_random, 2048, 5000),
    ("bucket", "n2049", rop_random, 2049, 5000),
    ("bucket", "sweep", rop_random, "bucket+0", 1 << 20),
    ("bucket", "sweep+1", rop_random, "bucket+1", 1 << 20),
    ("bucket", "3M", rop_invalid(0), 3000000, 1 << 21),
    ("fb-hubsize", "3M-invalid5000", rop_invalid(5000), 3000000, 1 << 20),
]


@pytest.mark.gpu
@pytest.mark.parametrize("path,gen,N,R", [pytest.param(c[0], *c[2:], id="%s-%s" % c[:2]) for c in CSR_CASES])
def test_csr_build_exact(cuda, path, gen, N, R):
    """dm_csr_build: point ids grouped by region, ascending inside a region (the stable order), points without a
    region (< 0 or >= n_regions) last; offsets[r] = first position of region r for r <= n_regions."""
    L = lib()
    N = resolve_n(N, sms())
    rng = np.random.default_rng(N + R)
    rop = gen(rng, N, R)
    key = np.where((rop >= 0) & (rop < R), rop, R).astype(np.int64)
    rule, misc = bucket_rule(key, R + 1)
    assert rule == path
    order = np.argsort(key, kind="stable").astype(np.int32)
    offs = np.searchsorted(key[order], np.arange(R + 1), side="left").astype(np.int64)
    query = L.dm_csr_workspace_bytes(N, R)
    import torch
    rop_d = torch.from_numpy(rop).cuda()
    prev = None
    for _ in range(2):
        off, ids = Guarded((R + 1) * 8), Guarded(N * 4)
        ws = workspace(query)
        L.check(L.dm_csr_build(rop_d.data_ptr(), N, R, off.ptr(), ids.ptr(), ws.data_ptr(), query, None), "dm_csr_build")
        sync()
        check_probe(ws, query - 256, misc)
        go, gi = off.get(np.int64), ids.get(np.int32)
        assert np.array_equal(gi, order) and np.array_equal(go, offs)
        assert off.intact() and ids.intact()
        if prev is not None:
            assert np.array_equal(prev[0], go) and np.array_equal(prev[1], gi)
        prev = (go.copy(), gi.copy())


def forest_random(rng, R):
    comp = rng.integers(0, R // 3, R)
    first = np.full(R // 3, R)
    np.minimum.at(first, comp, np.arange(R))
    return first[comp].astype(np.int32)


def forest_hubs(size, count=1):
    """`count` components of one root and `size` absorbed members each, then pairs."""
    def g(rng, R):
        parent = np.arange(R, dtype=np.int32)
        for c in range(count):
            parent[c * (size + 1):(c + 1) * (size + 1)] = c * (size + 1)
        rest = np.arange(count * (size + 1), R - 1, 2)
        parent[rest + 1] = rest
        return parent
    return g


MERGE_CASES = [
    ("bucket", "random", forest_random, 5000),
    ("bucket", "root48", forest_hubs(HUB_MIN), 5000),
    ("bucket-hubs", "root49", forest_hubs(HUB_MIN + 1), 5000),
    ("bucket-hubs", "root2048", forest_hubs(HUB_MAX_SORT), 5000),
    ("fb-hubsize", "root2049", forest_hubs(HUB_MAX_SORT + 1), 5000),
    ("bucket-hubs", "roots1024x49", forest_hubs(HUB_MIN + 1, HUB_CAP), 52000),
    ("fb-hubcount", "roots1025x49", forest_hubs(HUB_MIN + 1, HUB_CAP + 1), 52000),
]


@pytest.mark.gpu
@pytest.mark.parametrize("path,gen,R", [pytest.param(c[0], *c[2:], id="%s-%s" % c[:2]) for c in MERGE_CASES])
def test_merge_apply_member_sort_exact(cuda, path, gen, R):
    """dm_merge_apply sorts its (root, member) list by root and member (the bucket sort by the high half, no values):
    the list at the start of its workspace must be that sorted list, with its length in the int64 that ends the layout.
    Counts, areas and perimeters of the absorbed regions go to their roots."""
    L = lib()
    rng = np.random.default_rng(R)
    parent = gen(rng, R)
    x = np.nonzero(parent != np.arange(R))[0]
    want = np.sort(pack(parent[x], x))
    rule, misc = bucket_rule(parent[x], R)
    assert rule == path
    cnt0 = rng.integers(1, 100, R).astype(np.int32)
    area0 = rng.integers(1, 1000, R).astype(np.int64)
    per0 = rng.integers(1, 1000, R).astype(np.int64)
    cnt_w, area_w, per_w = cnt0.copy(), area0.copy(), per0.copy()
    np.add.at(cnt_w, parent[x], cnt0[x])
    np.add.at(area_w, parent[x], area0[x])
    np.add.at(per_w, parent[x], per0[x])
    query = L.dm_merge_apply_workspace_bytes(R)
    import torch
    T = lambda a: torch.from_numpy(a).cuda()
    prev = None
    for _ in range(2):
        par_d, alive = T(parent), T(np.ones(R, np.uint8))
        changed = T(np.zeros(R, np.uint8))
        s = T(np.zeros((R, 1), np.float32))
        cnt, area, per = T(cnt0), T(area0), T(per0)
        nm = Guarded(8)
        ws = workspace(query)
        L.check(L.dm_merge_apply(par_d.data_ptr(), alive.data_ptr(), changed.data_ptr(), s.data_ptr(), cnt.data_ptr(),
                                 area.data_ptr(), per.data_ptr(), R, 1, nm.ptr(), ws.data_ptr(), query, None),
                "dm_merge_apply")
        sync()
        check_probe(ws, query - 512, misc)
        n_list = int(ws[query - 256:query - 248].cpu().numpy().view(np.int64)[0])
        got = ws[:8 * n_list].cpu().numpy().view(U64)
        assert n_list == x.size and int(nm.get(np.int64)[0]) == x.size and nm.intact()
        assert np.array_equal(got, want)
        assert np.array_equal(cnt.cpu().numpy(), cnt_w) and np.array_equal(area.cpu().numpy(), area_w)
        assert np.array_equal(per.cpu().numpy(), per_w)
        assert np.array_equal(alive.cpu().numpy(), (parent == np.arange(R)).astype(np.uint8))
        if prev is not None:
            assert np.array_equal(prev, got)
        prev = got.copy()


# ------------------------------------------------------------------------------------------
# scan
# ------------------------------------------------------------------------------------------
SCAN_GUARD = 8192                # the unclamped scan reached up to 2047 items (8188 bytes) past the capacity

SCAN_CASES = [
    ("n0", 0, 3000, "small"), ("n1", 1, 3000, "small"), ("n2047", 2047, 2047, "small"), ("n2048", 2048, 2048, "small"),
    ("n2049", 2049, 2049, "small"), ("garbage", 2500, 7000, "small"), ("wrap", 1000, 1000, "wrap"),
    ("wrap-3M", 3000000, 3000123, "wrap"), ("tiles1024", 1024 * 2048, 1024 * 2048, "small"),
    ("tiles1025", 1024 * 2048 + 1, 1024 * 2048 + 1, "small"),
    ("over-cap+1", 3000 + 1, 3000, "small"), ("over-cap+1047", 3000 + 1047, 3000, "small"),
    ("over-cap+2047", 3000 + 2047, 3000, "wrap"), ("over-cap-3M+2047", 3000000 + 2047, 3000000, "small"),
]


@pytest.mark.gpu
@pytest.mark.parametrize("n_dev,cap,vals", [pytest.param(*c[1:], id=c[0]) for c in SCAN_CASES])
def test_scan_exclusive_u32_exact(cuda, n_dev, cap, vals):
    """dm_scan_exclusive_u32 over n = min(*n_dev, capacity) items: out[i] = in[0] + ... + in[i-1] mod 2^32 for i < n,
    the total mod 2^32; nothing at or past n is written, nothing past the capacity read.  The capacities 3000 and
    3000000 are not multiples of the 2048-item tile: a count above them made the last tile run past the capacity."""
    L = lib()
    rng = np.random.default_rng(n_dev + cap)
    n = min(n_dev, cap)
    if vals == "wrap":
        x = rng.integers(1 << 31, 1 << 32, cap, dtype=np.uint64).astype(np.uint32)
    else:
        x = rng.integers(0, 1000, cap).astype(np.uint32)
    ex, total = scan_ref(x[:n])
    o0 = rng.integers(0, 1 << 32, cap, dtype=np.uint64).astype(np.uint32)
    query = L.dm_scan_workspace_bytes(cap)
    prev = None
    for _ in range(2):
        xin = Guarded(cap * 4, x, SCAN_GUARD)
        out = Guarded(cap * 4, o0, SCAN_GUARD)
        nd = Guarded(8, np.array([n_dev], np.int64))
        tot = Guarded(8, np.array([-5], np.int64))
        ws = workspace(query)
        L.check(L.dm_scan_exclusive_u32(xin.ptr(), out.ptr(), nd.ptr(), cap, tot.ptr(), ws.data_ptr(), query, None),
                "dm_scan_exclusive_u32")
        sync()
        g = out.get(np.uint32)
        assert out.intact(), "the scan wrote past its capacity"
        assert np.array_equal(g[:n], ex) and np.array_equal(g[n:], o0[n:])
        assert int(tot.get(np.int64)[0]) == total
        assert np.array_equal(xin.get(np.uint32), x) and xin.intact() and nd.intact() and tot.intact()
        if prev is not None:
            assert np.array_equal(prev, g)
        prev = g.copy()
