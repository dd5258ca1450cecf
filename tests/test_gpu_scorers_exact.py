"""Edge scorers compared bit for bit: the pair-MLP (dm_score_mlp_bf16 / dm_mlp_forward_bf16) and the L2 scorer
(dm_score_l2, dm_euclidean_matrix) against float64 restatements, across their tiling and gather paths.

The inputs are built so that every product and every partial sum the kernels form is an integer below 2^24.  fp32
summation is then exact in any order, and a kernel must equal the float64 restatement exactly; the restatement rounds
to bf16 exactly where the kernel does.  A swapped or dropped K column, a row gathered from its neighbour, a wrong
rounding mode or one missing bias entry each change the result, so none can hide behind a tolerance.

Pair-MLP recipe (the builders assert it):
  x in [-2, 2]; each W1 row has at most 64 entries of +-1 and b1 = 2 nnz(row), so h1 in [0, 256] (exact in bf16);
  each W2 row has at most 8 entries of +-1 and b2 = 256 nnz(row), so h2 in [0, 4096] -- most h2 values are rounded to
  bf16 for layer 3, ties included, which exercises round-to-nearest-even; W3 in {-1, 0, 1} and b3 puts about half the
  logits below zero, where leaky_relu takes the fp32 product 0.01f * x of an exact x.
Layers 1 and 2 stay non-negative on purpose: bf16(0.01 x) feeding another layer cannot be made exact.  The negative
slope inside the network stays covered by the tolerance tests of test_gpu_mlp.py.

L2 recipe: means are integers in [-8, 8] and D <= 1000, so |x|^2, x.y and |x|^2 + |y|^2 - 2 x.y are exact and the
correctly rounded __fsqrt_rn must equal np.sqrt of the fp32 value.

Each GPU case asserts which kernel path its inputs select (vec4 or scalar gather, vec or scalar L2 kernel, tiles per
CTA), restating the selection rule of csrc/mlp.cu and csrc/score.cu; the test ids name the path.
"""
import numpy as np
import pytest

from oracle import oracle_np as o

M_TILE, KC, STAGES = 128, 64, 3                 # pair-MLP tile rows, K columns per ring chunk, ring stages
SENTINEL = np.array([0xDEADBEEF], np.uint32).view(np.float32)[0]


def T(x, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def num_sms():
    from deepmerge_b200._lib import lib
    n = lib().dm_num_sms()
    assert n > 0
    return n


def same(got, want):
    """Bitwise equality, NaN matching NaN whatever its payload."""
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    assert got.shape == want.shape
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan), "NaN rows differ"
    assert np.array_equal(got[~nan].view(np.uint32), want[~nan].view(np.uint32)), \
        "%d of %d values differ" % (int((got[~nan] != want[~nan]).sum()), int((~nan).sum()))


def offset_copy(t):
    """The same values in a contiguous tensor whose base is 4 bytes past a 16-byte boundary."""
    import torch
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


# ------------------------------------------------------------------------------------------
# float64 restatements
# ------------------------------------------------------------------------------------------
def bf16_rne(v):
    """float64 -> nearest bf16 value (8 significant bits), ties to even."""
    m, e = np.frexp(np.asarray(v, np.float64))
    return np.ldexp(np.round(m * 256.0), e - 8)


def bf16_trunc(v):
    """bf16 by truncation: the rounding mode the kernel must NOT use."""
    m, e = np.frexp(np.asarray(v, np.float64))
    return np.ldexp(np.trunc(m * 256.0), e - 8)


def lrelu(v):
    """fmaxf(x, 0.01f * x) on an fp32 x: the negative side is one fp32 product."""
    v32 = v.astype(np.float32)
    return np.where(v >= 0, v, (v32 * np.float32(0.01)).astype(np.float64))


def mlp_ref(x, W1, b1, W2, b2, W3, b3, rnd=bf16_rne):
    """The pair-MLP in float64: operands rounded to bf16 where the kernel rounds them -> (o, h2) fp32."""
    f = lambda a: np.asarray(a, np.float64)
    h1 = lrelu(rnd(f(x)) @ rnd(f(W1)).T + f(b1))
    h2 = lrelu(rnd(h1) @ rnd(f(W2)).T + f(b2))
    out = lrelu(rnd(h2) @ rnd(f(W3)).T + f(b3))
    return out.astype(np.float32), h2.astype(np.float32)


def exact_int(a, bound):
    a = np.asarray(a, np.float64)
    assert np.array_equal(a, np.round(a)) and np.abs(a).max(initial=0) < bound


# ------------------------------------------------------------------------------------------
# builders
# ------------------------------------------------------------------------------------------
def sparse_pm1(rng, rows, cols, max_nnz):
    """rows x cols of {-1, 0, +1}, at most max_nnz non-zeros per row."""
    W = np.zeros((rows, cols), np.float32)
    nnz = rng.integers(0, min(max_nnz, cols) + 1, rows)
    for r in range(rows):
        c = rng.choice(cols, nnz[r], replace=False)
        W[r, c] = rng.choice(np.array([-1.0, 1.0], np.float32), nnz[r])
    return W, nnz


def mlp_weights(rng, x, hidden, n_out):
    """Weights for x (finite rows, integers in [-2, 2]) under which the network's arithmetic is exact."""
    K = x.shape[1]
    exact_int(x, 3)
    W1, nnz1 = sparse_pm1(rng, hidden, K, 64)
    b1 = (2 * nnz1).astype(np.float32)
    W2, nnz2 = sparse_pm1(rng, hidden, hidden, 8)
    b2 = (256 * nnz2).astype(np.float32)
    W3 = rng.integers(-1, 2, (n_out, hidden)).astype(np.float32)
    x64 = x.astype(np.float64)
    a1 = x64 @ W1.T.astype(np.float64) + b1
    exact_int(a1, 257)
    assert a1.min(initial=0) >= 0                                   # h1 in [0, 256]: lrelu is the identity, bf16 exact
    assert np.array_equal(bf16_rne(a1), a1)
    a2 = a1 @ W2.T.astype(np.float64) + b2
    exact_int(a2, 4097)
    assert a2.min(initial=0) >= 0                                   # h2 in [0, 4096]
    z = bf16_rne(a2) @ W3.T.astype(np.float64)
    exact_int(z, 1 << 24)                                           # every partial sum too: |terms| sum to < 2^24
    assert hidden * 4096 < (1 << 24)
    b3 = (-np.floor(np.median(z, axis=0)) if len(z) else np.zeros(n_out)).astype(np.float32)
    return [W1, b1, W2, b2, W3, b3]


def int_means(rng, R, D, lim):
    return rng.integers(-lim, lim + 1, (R, D)).astype(np.float32)


def edge_keys(rng, R, n):
    """n keys lo < hi over R regions; the first ones touch region R - 1 and ids above 2^17."""
    lo = rng.integers(0, R - 1, n)
    hi = rng.integers(lo + 1, R)
    fixed = [(R - 2, R - 1), (0, R - 1), (R // 2, R - 1)]
    if R > (1 << 17) + 2:
        fixed += [((1 << 17) + 1, R - 1), (1 << 17, (1 << 17) + 1)]
    for i, (a, b) in enumerate(fixed[:n]):
        lo[i], hi[i] = a, b
    return o.pack_keys(lo, hi)


def l2_ref(mean, keys):
    """float64 expanded distance of every edge, rounded once to fp32 before the correctly rounded sqrt."""
    lo, hi = o.unpack_keys(keys)
    M = mean.astype(np.float64)
    assert 64 * M.shape[1] < (1 << 24)                              # |x|^2, x.y and every partial sum stay exact
    G = M @ M.T                                                     # exact: integers far below 2^53
    v = G[lo, lo] + G[hi, hi] - 2 * G[lo, hi]
    return np.sqrt(np.maximum(v, 0).astype(np.float32))


# ------------------------------------------------------------------------------------------
# CPU: the premise, and that the exact comparison has teeth
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,K,hidden,n_out", [(300, 200, 250, 2), (64, 784, 256, 16), (50, 1, 1, 1), (70, 130, 65, 3),
                                                 (40, 1000, 129, 15)])
def test_exact_builders_premise_and_oracle(rows, K, hidden, n_out):
    rng = np.random.default_rng(rows * K + hidden)
    x = rng.integers(-2, 3, (rows, K)).astype(np.float32)
    W = mlp_weights(rng, x, hidden, n_out)
    want_o, want_h2 = mlp_ref(x, *W)
    got_o, got_h2 = o.mlp_forward_bf16(x, *W)
    assert np.array_equal(got_o, want_o) and np.array_equal(got_h2, want_h2)
    if rows * hidden >= 10000:
        h2 = want_h2.astype(np.float64)
        rounded = bf16_rne(h2) != h2
        tie = np.zeros_like(rounded)
        for s in range(1, 5):                                       # [128 step, 256 step) has bf16 step `step`
            step = 2.0 ** s
            tie |= (h2 >= 128 * step) & (h2 < 256 * step) & (np.mod(h2, step) == step / 2)
        assert rounded.mean() > 0.5 and tie.sum() > 0               # layer 3's operand rounding is exercised, ties too
        assert (want_o < 0).mean() > 0.2 and (want_o > 0).mean() > 0.2


def test_exact_comparison_rejects_subtle_mutations():
    rng = np.random.default_rng(5)
    x = rng.integers(-2, 3, (1000, 200)).astype(np.float32)
    W = mlp_weights(rng, x, 250, 2)
    want = o.mlp_forward_bf16(x, *W)
    eq = lambda a, b: np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert eq(mlp_ref(x, *W), want)
    assert not eq(mlp_ref(x, *W, rnd=bf16_trunc), want)
    j = int(np.nonzero(W[3])[0][0])
    b2 = W[3].copy()
    b2[j] = 0
    assert not eq(mlp_ref(x, W[0], W[1], W[2], b2, W[4], W[5]), want)


def test_l2_builder_premise_and_oracle():
    rng = np.random.default_rng(3)
    for D in (1, 5, 132, 1000):
        mean = int_means(rng, 500, D, 8)
        keys = edge_keys(rng, 500, 2000)
        assert np.array_equal(o.score_l2(mean, keys), l2_ref(mean, keys))       # the fp32 oracle, any summation order


# ------------------------------------------------------------------------------------------
# GPU: pair-MLP case matrix
# ------------------------------------------------------------------------------------------
ROWS = {"1": lambda S: 1, "127": lambda S: 127, "128": lambda S: 128, "129": lambda S: 129,
        "S128": lambda S: S * M_TILE, "S128+1": lambda S: S * M_TILE + 1, "3S128+77": lambda S: 3 * S * M_TILE + 77}
TPC = {"1": (1, 1), "S128": (1, 1), "127": (1, 1), "128": (1, 1), "129": (1, 1), "S128+1": (1, 2), "3S128+77": (3, 4)}
R_EDGE = (1 << 17) + 3001


def tiles_per_cta(rows, S):
    """(fewest, most) tiles a CTA of the persistent grid walks: grid = min(tiles, SMs), tiles strided by the grid."""
    tiles = -(-rows // M_TILE)
    grid = max(1, min(tiles, S))
    return tiles // grid, -(-tiles // grid)


def gather_path(D, K, ld, ptr):
    """The producer warps' choice in pair_mlp_kernel: 128-bit gathers only when every row piece is 16-byte aligned."""
    return "vec4" if D % 4 == 0 and K % 4 == 0 and ld % 4 == 0 and ptr % 16 == 0 else "scalar"


def mlp_case_id(mode, F, rows, hidden, n_out, gather):
    K = 2 * F if mode == "edge" else F
    nk1 = -(-K // KC)
    return "%s-%s%d-rows%s-h%d-o%d-%s-nk%d-ring%d-tpc%d..%d" % (mode, "D" if mode == "edge" else "K", F, rows, hidden,
                                                                  n_out, gather, nk1, (nk1 + 4) % STAGES, *TPC[rows])


# (features per endpoint D, rows, hidden, n_out, gather).  Pairwise over the axes, not the cross-product; the rows of
# 3 to 4 tiles per CTA run with every ring residue (nk1 + 4) mod 3 on both gathers' sides.
EDGE_CASES = [
    (100, "3S128+77", 250, 2, "vec4"),      # the bench shape: nk1 4, ring residue 2
    (64, "3S128+77", 129, 3, "vec4"),       # nk1 2, residue 0
    (96, "3S128+77", 65, 16, "vec4"),       # nk1 3, residue 1
    (7, "3S128+77", 31, 15, "scalar"),      # nk1 1, residue 2
    (33, "S128+1", 256, 1, "scalar"),
    (32, "1", 31, 16, "vec4"),
    (32, "S128", 128, 2, "vec4"),
    (7, "127", 64, 3, "scalar"),
    (33, "128", 250, 15, "scalar"),
    (100, "129", 1, 1, "vec4"),
    (96, "1", 256, 2, "vec4"),
    (64, "128", 1, 16, "vec4"),
    (100, "S128+1", 65, 16, "vec4"),
    (7, "129", 129, 2, "scalar"),
    (33, "1", 128, 3, "scalar"),
    (64, "127", 250, 15, "vec4"),
]
DENSE_CASES = [
    (65, "3S128+77", 31, 3, "scalar"),      # nk1 2, residue 0
    (129, "3S128+77", 64, 15, "scalar"),    # nk1 3, residue 1
    (1, "3S128+77", 250, 16, "scalar"),     # nk1 1, residue 2
    (128, "3S128+77", 129, 1, "vec4"),      # nk1 2, residue 0
    (200, "3S128+77", 256, 2, "vec4"),      # nk1 4, residue 2
    (1, "1", 1, 1, "scalar"),
    (63, "127", 256, 2, "scalar"),
    (63, "S128+1", 1, 15, "scalar"),
    (65, "S128", 256, 16, "scalar"),
    (129, "128", 31, 2, "scalar"),
    (784, "129", 250, 2, "vec4"),           # nk1 13
    (1000, "128", 65, 1, "vec4"),           # nk1 16
    (784, "1", 128, 16, "vec4"),
    (1000, "127", 1, 3, "vec4"),
    (200, "129", 64, 15, "vec4"),
]


def packed(cuda, W):
    from deepmerge_b200 import PackedMLP
    return PackedMLP(*[T(w, cuda) for w in W])


def edge_inputs(rng, D, E, R=R_EDGE):
    mean = int_means(rng, R, D, 2)
    keys = edge_keys(rng, R, E)
    return mean, keys


@pytest.mark.gpu
@pytest.mark.parametrize("D,rows,hidden,n_out,gather", [pytest.param(*c, id=mlp_case_id("edge", *c)) for c in EDGE_CASES])
def test_score_mlp_exact(cuda, D, rows, hidden, n_out, gather):
    from deepmerge_b200 import score_mlp
    S = num_sms()
    E = ROWS[rows](S)
    assert tiles_per_cta(E, S) == TPC[rows]
    rng = np.random.default_rng(D * 1000 + E + hidden)
    mean, keys = edge_inputs(rng, D, E)
    x = o.pair_features(mean, keys)
    W = mlp_weights(rng, x, hidden, n_out)
    want_o, want_h2 = mlp_ref(x, *W)
    mean_t = T(mean, cuda)
    assert gather_path(D, 2 * D, D, mean_t.data_ptr()) == gather
    got_o, got_h2 = score_mlp(mean_t, T(keys.view(np.int64), cuda), packed(cuda, W), want_h2=True, check=True)
    same(got_h2.cpu().numpy(), want_h2)
    same(got_o.cpu().numpy(), want_o)


@pytest.mark.gpu
@pytest.mark.parametrize("K,rows,hidden,n_out,gather", [pytest.param(*c, id=mlp_case_id("dense", *c)) for c in DENSE_CASES])
def test_mlp_forward_exact(cuda, K, rows, hidden, n_out, gather):
    from deepmerge_b200 import mlp_forward
    S = num_sms()
    B = ROWS[rows](S)
    assert tiles_per_cta(B, S) == TPC[rows]
    rng = np.random.default_rng(K * 1000 + B + hidden)
    x = rng.integers(-2, 3, (B, K)).astype(np.float32)
    W = mlp_weights(rng, x, hidden, n_out)
    want_o, want_h2 = mlp_ref(x, *W)
    x_t = T(x, cuda)
    assert gather_path(K, K, K, x_t.data_ptr()) == gather
    got_o, got_h2 = mlp_forward(x_t, packed(cuda, W), want_h2=True, check=True)
    same(got_h2.cpu().numpy(), want_h2)
    same(got_o.cpu().numpy(), want_o)


# ------------------------------------------------------------------------------------------
# GPU: pair-MLP contract
# ------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def bench_shape_case(cuda):
    """D = 100, hidden 250, n_out 2 over 3 to 4 tiles per CTA, with its float64 result."""
    S = num_sms()
    E = ROWS["3S128+77"](S)
    rng = np.random.default_rng(11)
    mean, keys = edge_inputs(rng, 100, E)
    x = o.pair_features(mean, keys)
    W = mlp_weights(rng, x, 250, 2)
    return mean, keys, W, mlp_ref(x, *W)


@pytest.mark.gpu
def test_score_mlp_row_count_below_capacity(cuda, bench_shape_case):
    """The merge loop passes the live edge count on the device and the capacity on the host: rows at and past the
    count keep what the output held, bit for bit, and a count of 0 writes nothing."""
    import torch
    from deepmerge_b200 import score_mlp
    mean, keys, W, (want_o, _) = bench_shape_case
    S = num_sms()
    cap = keys.shape[0]
    mlp = packed(cuda, W)
    mean_t, keys_t = T(mean, cuda), T(keys.view(np.int64), cuda)
    for n in (0, 1, 129, S * M_TILE + 1, cap - 1):
        out = torch.full((cap, 2), float(SENTINEL), dtype=torch.float32, device=cuda)
        nd = torch.tensor([n], dtype=torch.int64, device=cuda)
        got, _ = score_mlp(mean_t, keys_t, mlp, n_edges_dev=nd, out=out, check=True)
        assert got.data_ptr() == out.data_ptr()
        g = out.cpu().numpy()
        same(g[:n], want_o[:n])
        assert np.array_equal(g[n:].view(np.uint32), np.full((cap - n, 2), 0xDEADBEEF, np.uint32)), n


@pytest.mark.gpu
def test_score_mlp_without_h2_and_repeated(cuda, bench_shape_case):
    """want_h2=False gives the same logits; two calls on one packed blob give identical results."""
    from deepmerge_b200 import score_mlp
    mean, keys, W, (want_o, want_h2) = bench_shape_case
    mlp = packed(cuda, W)
    mean_t, keys_t = T(mean, cuda), T(keys.view(np.int64), cuda)
    a_o, a_h2 = score_mlp(mean_t, keys_t, mlp, want_h2=True, check=True)
    b_o, b_h2 = score_mlp(mean_t, keys_t, mlp, want_h2=False, check=True)
    c_o, c_h2 = score_mlp(mean_t, keys_t, mlp, want_h2=True, check=True)
    assert b_h2 is None and int(mlp.status.item()) == 0
    for got in (a_o, b_o, c_o):
        same(got.cpu().numpy(), want_o)
    same(a_h2.cpu().numpy(), want_h2)
    same(c_h2.cpu().numpy(), want_h2)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [100, 64])
def test_score_mlp_misaligned_mean(cuda, D):
    """A contiguous mean whose base is 4 bytes off 16-byte alignment takes the scalar gather even though D % 4 == 0,
    and gives what the aligned copy gives.  The same for dense rows."""
    from deepmerge_b200 import mlp_forward, score_mlp
    S = num_sms()
    E = S * M_TILE + 1
    rng = np.random.default_rng(D)
    mean, keys = edge_inputs(rng, D, E, R=(1 << 17) + 17)
    x = o.pair_features(mean, keys)
    W = mlp_weights(rng, x, 129, 3)
    want_o, want_h2 = mlp_ref(x, *W)
    mlp = packed(cuda, W)
    keys_t = T(keys.view(np.int64), cuda)
    aligned = T(mean, cuda)
    shifted = offset_copy(aligned)
    assert gather_path(D, 2 * D, D, aligned.data_ptr()) == "vec4"
    assert gather_path(D, 2 * D, D, shifted.data_ptr()) == "scalar"
    for m in (aligned, shifted):
        got_o, got_h2 = score_mlp(m, keys_t, mlp, want_h2=True, check=True)
        same(got_o.cpu().numpy(), want_o)
        same(got_h2.cpu().numpy(), want_h2)
    # dense mode, K = 2 D rows of the same features
    x_t = T(x, cuda)
    xs = offset_copy(x_t)
    assert gather_path(2 * D, 2 * D, 2 * D, x_t.data_ptr()) == "vec4"
    assert gather_path(2 * D, 2 * D, 2 * D, xs.data_ptr()) == "scalar"
    for xx in (x_t, xs):
        got_o, got_h2 = mlp_forward(xx, mlp, want_h2=True, check=True)
        same(got_o.cpu().numpy(), want_o)
        same(got_h2.cpu().numpy(), want_h2)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [100, 7])
def test_score_mlp_nan_rows(cuda, D):
    """A region without sample points has a NaN mean: every logit of its edges is NaN (the merge rule never selects
    them), and the other rows of the same tiles are exact."""
    from deepmerge_b200 import score_mlp
    rng = np.random.default_rng(D + 1)
    E = 3 * M_TILE + 5
    R = (1 << 17) + 77
    mean, keys = edge_inputs(rng, D, E, R=R)
    lo, hi = o.unpack_keys(keys)
    bad = np.unique(np.r_[hi[0], lo[[5, 70, 127, 128, 300]], hi[[200, E - 1]]])   # R - 1 among them
    x = o.pair_features(mean, keys)
    W = mlp_weights(rng, x, 250, 5)
    want_o, want_h2 = mlp_ref(x, *W)
    mean_nan = mean.copy()
    mean_nan[bad] = np.nan
    nan_row = np.isin(lo, bad) | np.isin(hi, bad)
    assert nan_row.sum() >= len(bad) and (~nan_row).sum() > E // 2
    got_o, got_h2 = score_mlp(T(mean_nan, cuda), T(keys.view(np.int64), cuda), packed(cuda, W), want_h2=True, check=True)
    got_o, got_h2 = got_o.cpu().numpy(), got_h2.cpu().numpy()
    assert np.isnan(got_o[nan_row]).all()
    same(got_o[~nan_row], want_o[~nan_row])
    same(got_h2[~nan_row], want_h2[~nan_row])


# ------------------------------------------------------------------------------------------
# GPU: L2 scorer and distance matrix
# ------------------------------------------------------------------------------------------
R_L2 = 1500


def l2_kernel(D, ptr):
    """dm_score_l2's choice: the vec kernel for D % 4 == 0 on a 16-byte aligned mean, else the scalar one."""
    return "vec" if D % 4 == 0 and ptr % 16 == 0 else "scalar"


def l2_id(D, offset):
    k = "scalar" if offset or D % 4 else "vec%dtrip" % -(-D // 128)
    return "D%d-%s-%s" % (D, "offset4" if offset else "aligned", k)


L2_CASES = [(D, off) for D in (1, 3, 4, 5, 100, 128, 129, 132, 260, 1000) for off in (False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("D,offset", [pytest.param(D, off, id=l2_id(D, off)) for D, off in L2_CASES])
def test_score_l2_exact(cuda, D, offset):
    """dm_score_l2 through the raw ABI: every edge bit for bit, past one grid-stride sweep of either kernel and at
    E = 1; a device count below the capacity leaves the tail alone; `rescore` leaves edges without a flagged endpoint
    alone; NaN means give NaN scores."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    S = num_sms()
    rng = np.random.default_rng(D * 2 + offset)
    mean = int_means(rng, R_L2, D, 8)
    bad = rng.choice(R_L2 - 1, 6, replace=False)
    mean[bad] = np.nan
    norm2 = np.einsum("ij,ij->i", mean.astype(np.float64), mean.astype(np.float64)).astype(np.float32)
    mean_t = T(mean, cuda)
    if offset:
        mean_t = offset_copy(mean_t)
    kernel = l2_kernel(D, mean_t.data_ptr())
    assert kernel == ("scalar" if offset or D % 4 else "vec")
    norm2_t = T(norm2, cuda)
    sweep = 4 * 8 * 8 * S if kernel == "vec" else 8 * 8 * S          # edges one pass of the capped grid covers
    flags = (rng.random(R_L2) < 0.1).astype(np.uint8)
    flags_t = T(flags, cuda)
    for E in (1, 4 * 8 * 8 * S + 123):
        keys = edge_keys(rng, R_L2, E)
        want = l2_ref(np.nan_to_num(mean), keys)
        lo, hi = o.unpack_keys(keys)
        want[np.isin(lo, bad) | np.isin(hi, bad)] = np.nan
        if E > 1:
            assert E > sweep and np.isnan(want).sum() > 0
        keys_t = T(keys.view(np.int64), cuda)

        def run(n, rescore):
            sc = torch.full((E,), float(SENTINEL), dtype=torch.float32, device=cuda)
            nd = torch.tensor([n], dtype=torch.int64, device=cuda)
            L.check(L.dm_score_l2(mean_t.data_ptr(), norm2_t.data_ptr(), D, keys_t.data_ptr(), nd.data_ptr(), E,
                                  rescore.data_ptr() if rescore is not None else None, sc.data_ptr(), None), "dm_score_l2")
            return sc.cpu().numpy()

        same(run(E, None), want)
        n = E // 2 + 3 if E > 1 else 0
        got = run(n, None)
        same(got[:n], want[:n])
        assert np.all(got[n:].view(np.uint32) == 0xDEADBEEF)
        got = run(E, flags_t)
        hit = (flags[lo] != 0) | (flags[hi] != 0)
        same(got[hit], want[hit])
        assert np.all(got[~hit].view(np.uint32) == 0xDEADBEEF)
        if E > 1:
            assert hit.sum() > 0 and (~hit).sum() > 0


@pytest.mark.gpu
@pytest.mark.parametrize("p", [1, 13, 100, 129])
def test_euclidean_matrix_exact(cuda, p):
    """dm_euclidean_matrix on 200 x 300 outputs (several sweeps of its capped grid), bit for bit, nothing written past
    the n x m outputs."""
    import torch
    from deepmerge_b200._lib import lib
    L = lib()
    n, m = 200, 300
    assert n * m > 2 * 8 * 8 * num_sms()
    rng = np.random.default_rng(p)
    X, Y = int_means(rng, n, p, 8), int_means(rng, m, p, 8)
    X64, Y64 = X.astype(np.float64), Y.astype(np.float64)
    v = (X64 * X64).sum(1)[:, None] + (Y64 * Y64).sum(1)[None, :] - 2 * X64 @ Y64.T
    want = np.sqrt(np.maximum(v, 0).astype(np.float32))
    out = torch.full((n * m + 37,), float(SENTINEL), dtype=torch.float32, device=cuda)
    Xt, Yt = T(X, cuda), T(Y, cuda)
    L.check(L.dm_euclidean_matrix(Xt.data_ptr(), Yt.data_ptr(), n, m, p, out.data_ptr(), None), "dm_euclidean_matrix")
    got = out.cpu().numpy()
    same(got[:n * m].reshape(n, m), want)
    assert np.all(got[n * m:].view(np.uint32) == 0xDEADBEEF)
