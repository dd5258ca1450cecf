"""GPU: R8 pair-MLP on tcgen05 (dm_score_mlp_bf16 / dm_mlp_forward_bf16) against the executed-reference
golden vectors (Nets.MLP, fp32) and the oracle's bf16-operand restatement.

Tolerances.  The kernel rounds every GEMM operand (x, h1, h2, W*) to bf16 (8-bit mantissa, relative
rounding error 2^-9) and accumulates in fp32.  Against the oracle's mlp_forward_bf16, which rounds the
same operands, the only differences are the fp32 summation order and the bf16 roundings of h1 / h2 that
flip when a pre-activation sits within that order noise of a rounding boundary: |diff| <= 2e-2 * scale
is asserted, with scale = max |activation| of the layer.  Against the fp32 reference the operand rounding
itself shows: |diff| <= 5e-2 * scale.  Merge decisions (argmax of the two logits) must agree wherever
the oracle's logit margin exceeds the bf16 tolerance.
"""
import os

import numpy as np
import pytest

from oracle import golden
from oracle import oracle_np as o

pytestmark = pytest.mark.gpu


def T(x, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(x)).to(dev)


def close(got, want, tol):
    scale = max(1e-6, float(np.abs(want).max()))
    err = float(np.abs(got - want).max())
    assert err <= tol * scale, (err, scale)


@pytest.mark.parametrize("name", ["mlp_pair.npz", "mlp784.npz"])
def test_mlp_forward_against_reference_golden(cuda, golden_dir, name):
    from deepmerge_b200.Nets import MLP
    import torch
    m = golden.load(os.path.join(golden_dir, name))
    n_in, hidden, n_out = m["fc1_weight"].shape[1], m["fc1_weight"].shape[0], m["fc3_weight"].shape[0]
    net = MLP((n_in, hidden, n_out)).to(cuda)
    net.load_state_dict({k: torch.from_numpy(m[k.replace(".", "_")]) for k in
                         ("fc1.weight", "fc1.bias", "fc2.weight", "fc2.bias", "fc3.weight", "fc3.bias")})
    fc3, fc2 = net(T(m["x"], cuda))
    assert fc3.shape == m["fc3"].shape and fc2.shape == m["fc2"].shape
    W = [m[k] for k in ("fc1_weight", "fc1_bias", "fc2_weight", "fc2_bias", "fc3_weight", "fc3_bias")]
    ob, h2b = o.mlp_forward_bf16(m["x"], *W)
    close(fc2.cpu().numpy(), h2b, 2e-2)
    close(fc3.cpu().numpy(), ob, 2e-2)
    close(fc2.cpu().numpy(), m["fc2"], 5e-2)           # the fp32 reference itself (Nets.MLP executed)
    close(fc3.cpu().numpy(), m["fc3"], 5e-2)


@pytest.mark.parametrize("E,D,hidden,n_out", [(1, 100, 250, 2), (127, 100, 250, 2), (128, 100, 250, 2), (1000, 100, 250, 2),
                                              (40000, 100, 250, 2), (300, 16, 64, 3), (513, 33, 256, 16), (200, 7, 5, 1)])
def test_score_mlp_on_edges(cuda, E, D, hidden, n_out):
    from deepmerge_b200 import PackedMLP, score_mlp
    rng = np.random.default_rng(E + D)
    R = max(2, E // 3 + 2)
    mean = rng.standard_normal((R, D)).astype(np.float32)
    lo = rng.integers(0, R - 1, size=E)
    hi = np.minimum(R - 1, lo + 1 + rng.integers(0, 5, size=E))
    keys = o.pack_keys(lo, hi)
    s = lambda *sh: (rng.standard_normal(sh) / np.sqrt(sh[-1])).astype(np.float32)
    W = [s(hidden, 2 * D), s(hidden), s(hidden, hidden), s(hidden), s(n_out, hidden), s(n_out)]
    mlp = PackedMLP(*[T(w, cuda) for w in W])
    got_o, got_h2 = score_mlp(T(mean, cuda), T(keys.view(np.int64), cuda), mlp, want_h2=True)
    want_o, want_h2 = o.mlp_forward_bf16(o.pair_features(mean, keys), *W)
    close(got_h2.cpu().numpy(), want_h2, 2e-2)
    close(got_o.cpu().numpy(), want_o, 2e-2)
    if n_out >= 2:                                     # identical decisions outside the tolerance band
        margin = np.abs(want_o[:, 1] - want_o[:, 0])
        sure = margin > 4e-2 * max(1e-6, float(np.abs(want_o).max()))
        g = got_o.cpu().numpy()
        assert np.array_equal((g[:, 1] > g[:, 0])[sure], (want_o[:, 1] > want_o[:, 0])[sure])


def test_score_mlp_rejects_bad_shapes(cuda):
    from deepmerge_b200 import PackedMLP, score_mlp
    import torch
    z = lambda *s: torch.zeros(*s, device=cuda)
    with pytest.raises(ValueError):
        PackedMLP(z(300, 8), z(300), z(300, 300), z(300), z(2, 300), z(2))        # hidden > 256
    mlp = PackedMLP(z(8, 6), z(8), z(8, 8), z(8), z(2, 8), z(2))
    with pytest.raises(ValueError):
        score_mlp(z(4, 5), torch.zeros(1, dtype=torch.int64, device=cuda), mlp)   # in_features != 2 D


def test_merge_graph_with_mlp_matches_oracle(cuda):
    """The merge loop driven by the pair-MLP (argmax == 1 selects): final roots equal the oracle's when its
    decisions are taken from the same bf16 arithmetic, on a graph whose logit margins are wide."""
    from deepmerge_b200 import PackedMLP, merge_graph
    rng = np.random.default_rng(7)
    R, D, G = 400, 8, 40
    group = rng.integers(0, G, size=R)
    centre = rng.standard_normal((G, D)).astype(np.float32) * 4
    mean = (centre[group] + 0.01 * rng.standard_normal((R, D))).astype(np.float32)
    cnt = rng.integers(1, 5, size=R).astype(np.int32)
    sum_ = (mean * cnt[:, None]).astype(np.float32)
    lo = rng.integers(0, R - 1, size=1500)
    hi = np.minimum(R - 1, lo + 1 + rng.integers(0, 6, size=1500))
    keys = np.unique(o.pack_keys(lo, hi))
    blen = rng.integers(1, 9, size=keys.shape[0]).astype(np.uint32)
    area = rng.integers(5, 50, size=R).astype(np.int64)
    perim = area * 2
    # a hand-made "same object?" network: logit1 - logit0 = 4 - |mean_lo - mean_hi|_1-ish through lrelu units
    hidden = 2 * D
    W1 = np.zeros((hidden, 2 * D), np.float32)
    for d in range(D):
        W1[d, d], W1[d, D + d] = 1, -1                  # +(a-b)
        W1[D + d, d], W1[D + d, D + d] = -1, 1          # -(a-b)
    b1 = np.zeros(hidden, np.float32)
    W2 = np.eye(hidden, dtype=np.float32)
    b2 = np.zeros(hidden, np.float32)
    W3 = np.zeros((2, hidden), np.float32)
    W3[0] = 1.0                                         # logit0 ~ sum |a-b| (lrelu(x)+lrelu(-x) ~ |x|)
    b3 = np.array([0.0, 2.0], np.float32)               # logit1 = 2: merge iff sum|a-b| < ~2
    W = [W1, b1, W2, b2, W3, b3]
    want = o.merge_graph(sum_, cnt, area, perim, keys, blen, mlp=tuple(W), mlp_bf16=True)
    mlp = PackedMLP(*[T(w, cuda) for w in W])
    got = merge_graph(T(sum_, cuda), T(cnt, cuda), T(area, cuda), T(perim, cuda), T(keys.view(np.int64), cuda),
                      T(blen.view(np.int32), cuda), 0.0, mlp=mlp)
    assert np.array_equal(got.root.cpu().numpy(), want["root"])
    assert got.rounds == want["rounds"] and got.merges == want["merges"]
