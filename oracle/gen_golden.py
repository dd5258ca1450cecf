"""Generate tests/golden/*.npz by EXECUTING the reference's own code (TEST INFRASTRUCTURE).

Run in the build container only (needs /root/reference):  python -m oracle.gen_golden
The fixtures are committed; the GPU box never reads /root/reference.

Every block names the reference symbol it runs.  Nothing here is a restatement except
the pooling loop of test_for_shp (ExtractFeatures.py:188-216), which is transcribed
statement-for-statement around the *imported* Euclidean_distance because the original
hard-codes Windows paths, needs OGR/h5py and `break`s after the first edge (:223).
"""
from __future__ import annotations

import os
import sys
import random
import tempfile

import numpy as np
import torch

from . import golden, ref_shim

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def golden_euclid(ref, rng):
    ED = ref.ExtractFeatures.Euclidean_distance
    K, D = 96, 100
    X = rng.standard_normal((K, D)).astype(np.float32)
    Y = rng.standard_normal((K, D)).astype(np.float32)
    Y[16:32] = X[16:32] + (1e-4 * rng.standard_normal((16, D))).astype(np.float32)   # near-identical
    Y[32:40] = X[32:40]                                                             # identical
    X[40:44] = 0                                                                    # zero vector
    Y[44:48] = 0
    X[48:56] *= 100.0                                                               # large magnitude
    Y[48:56] *= 100.0
    X[56:64] = X[56:64] * 50 + 10
    Y[56:64] = X[56:64] + (1e-2 * rng.standard_normal((8, D))).astype(np.float32)
    d = np.stack([ED(X[i:i + 1], Y[i:i + 1])[0, 0] for i in range(K)])
    assert d.dtype == np.float32
    d2 = np.stack([ref.ExtractFeatures.MC_Lyu_2020(X[i:i + 1], Y[i:i + 1])[0, 0] for i in range(K)])
    assert np.array_equal(d, d2)
    Xm = rng.standard_normal((7, 13)).astype(np.float32)
    Ym = rng.standard_normal((5, 13)).astype(np.float32)
    np.savez(os.path.join(OUT, "euclid.npz"), X=X, Y=Y, d=d, Xm=Xm, Ym=Ym, Dm=ED(Xm, Ym))


def golden_pool_score(ref, rng):
    """test_for_shp's loop body, ExtractFeatures.py:164-222 minus IO and the break."""
    ED = ref.ExtractFeatures.Euclidean_distance
    R, D = 40, 100
    npts = rng.integers(1, 9, size=R)
    N = int(npts.sum())
    store = (rng.standard_normal((N, D)) + 3 * rng.standard_normal((1, D))).astype(np.float32)
    perm = rng.permutation(N)
    fields, pos = [], 0
    for r in range(R):
        fields.append(" ".join(str(int(t)) for t in perm[pos:pos + npts[r]]))
        pos += npts[r]
    E = 120
    left = rng.integers(0, R, size=E)
    right = (left + rng.integers(1, R, size=E)) % R
    simi = np.zeros(E, np.float64)
    means = np.zeros((R, D), np.float32)
    for e in range(E):
        left_poly_samples = fields[left[e]].split(' ')            # :178
        right_poly_samples = fields[right[e]].split(' ')          # :179
        out_left_data, out_right_data = [], []
        for m in range(0, len(left_poly_samples)):                # :190-198
            left_features = store[int(left_poly_samples[m])][np.newaxis, :]
            out_left_data = left_features if m == 0 else np.concatenate((out_left_data, left_features), axis=0)
        for n in range(0, len(right_poly_samples)):               # :199-207
            right_features = store[int(right_poly_samples[n])][np.newaxis, :]
            out_right_data = right_features if n == 0 else np.concatenate((out_right_data, right_features), axis=0)
        out_left_data = np.mean(out_left_data, axis=0)            # :211
        out_right_data = np.mean(out_right_data, axis=0)          # :212
        means[left[e]], means[right[e]] = out_left_data, out_right_data
        Dm = ED(out_left_data[np.newaxis, :], out_right_data[np.newaxis, :])   # :215
        simi[e] = float(Dm.max())                                 # :216-218 (OFTReal = float64)
    used = np.zeros(R, bool)
    used[left] = used[right] = True
    np.savez(os.path.join(OUT, "pool_score.npz"), store=store, fields=np.array(fields), left=left, right=right,
             simi=simi, means=means, used=used)


def golden_mlp(ref, rng):
    torch.manual_seed(0)
    m = ref.Nets.MLP().eval()
    x = torch.from_numpy(rng.standard_normal((32, 784)).astype(np.float32))
    with torch.no_grad():
        fc3, fc2 = m(x)
    sd = {k: v.numpy() for k, v in m.state_dict().items()}
    golden.save(os.path.join(OUT, "mlp784.npz"), x=x.numpy(), fc3=fc3.numpy(), fc2=fc2.numpy(),
             **{k.replace(".", "_"): v for k, v in sd.items()})
    # pair-MLP: the same class and forward code (Nets.py:28-35) with fc1/fc3 re-dimensioned
    torch.manual_seed(1)
    p = ref.Nets.MLP()
    p.fc1 = torch.nn.Linear(200, 250)
    p.fc3 = torch.nn.Linear(250, 2)
    p = p.eval()
    xp = torch.from_numpy(rng.standard_normal((300, 200)).astype(np.float32))
    with torch.no_grad():
        o, h2 = p(xp)
    sd = {k: v.numpy() for k, v in p.state_dict().items()}
    np.savez(os.path.join(OUT, "mlp_pair.npz"), x=xp.numpy(), fc3=o.numpy(), fc2=h2.numpy(),
             **{k.replace(".", "_"): v for k, v in sd.items()})


def golden_loss(ref, rng):
    B, D = 120, 100
    a = torch.from_numpy((0.1 * rng.standard_normal((B, D))).astype(np.float32)).requires_grad_(True)
    b = torch.from_numpy((0.1 * rng.standard_normal((B, D))).astype(np.float32)).requires_grad_(True)
    with torch.no_grad():
        b[:30] = a[:30] + 0.01                     # tiny d
    flag = torch.from_numpy(rng.integers(0, 2, size=B).astype(np.int64))
    out = {}
    for margin in (1.0, 2.5):
        crit = ref.Losses.Loss(margin, 0.1, 0)
        a.grad = b.grad = None
        loss = crit(a, b, flag)
        loss.backward()
        out[f"loss_{margin}"] = loss.detach().numpy()
        out[f"ga_{margin}"] = a.grad.numpy().copy()
        out[f"gb_{margin}"] = b.grad.numpy().copy()
    np.savez(os.path.join(OUT, "loss.npz"), a=a.detach().numpy(), b=b.detach().numpy(), flag=flag.numpy(), **out)


def golden_edge_reader(ref, rng):
    """PolygonConnectPointDataset.add_data, MyUtils2.py:155-193, on a fake lines.shp."""
    E = 64
    left = rng.integers(-1, 30, size=E)
    right = rng.integers(-1, 30, size=E)
    left[5] = right[5] = -1
    lines = ref_shim.FakeLayer([ref_shim.FakeFeature(i, {"LEFT_FID": int(left[i]), "RIGHT_FID": int(right[i])})
                                for i in range(E)])
    paths = {"X:\\tiles\\tileA.shp": ref_shim.FakeLayer([]), "X:\\tiles\\tileA\\lines.shp": lines,
             "X:\\tiles\\tileA\\PointsGCS.shp": ref_shim.FakeLayer([])}
    ref_shim.install_fake_drivers(ref, paths, {"X:\\img\\tileA.tif": ref_shim.FakeRaster(np.zeros((3, 8, 8), np.uint8))})
    ds = ref.MyUtils2.PolygonConnectPointDataset("X:\\img\\tileA.tif", "X:\\tiles\\tileA.shp",
                                                 "X:\\tiles\\tileA\\lines.shp", "X:\\tiles\\tileA\\PointsGCS.shp")
    rows = [ds[i] for i in range(len(ds))]
    np.savez(os.path.join(OUT, "edge_reader.npz"), left=left, right=right,
             out_fid=np.array([r[0] for r in rows]), out_name=np.array([r[1] for r in rows]),
             out_left=np.array([r[2] for r in rows]), out_right=np.array([r[3] for r in rows]))


def golden_pair_sampler(ref, rng):
    """MergingSegmensPairDataset.add_data, MyUtils1.py:236-295, with random.seed fixed."""
    R = 25
    npts = rng.integers(1, 6, size=R)
    fields, pos = [], 0
    for r in range(R):
        fields.append(" ".join(str(pos + k) for k in range(npts[r])))
        pos += int(npts[r])
    polys = ref_shim.FakeLayer([ref_shim.FakeFeature(r, {"PointID": fields[r]}) for r in range(R)])
    pts = ref_shim.FakeLayer([])
    pos_pairs = rng.integers(0, R, size=(40, 2))
    neg_pairs = rng.integers(0, R, size=(30, 2))
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for name, pairs in (("tileP.txt", pos_pairs), ("tileN.txt", neg_pairs)):
                with open(name, "w") as f:
                    for j, (a, b) in enumerate(pairs):
                        f.write(f"{j},{a},{b},0,0\n")                      # cols 1,2 are used (:231)
            layers = {}
            for t in ("tileP", "tileN"):
                layers[f"PF\\{t}.shp"] = polys
                layers[f"QF\\{t}\\PointsGCS.shp"] = pts
            rasters = {f"IF\\{t}.tif": ref_shim.FakeRaster(np.zeros((3, 8, 8), np.uint8)) for t in ("tileP", "tileN")}
            ref_shim.install_fake_drivers(ref, layers, rasters)
            ds = object.__new__(ref.MyUtils1.MergingSegmensPairDataset)
            ds.image_folder, ds.polygon_folder, ds.point_folder = "IF", "PF", "QF"
            ds.data, ds.point_dataset, ds.img_dataset, ds.layers = [], [], {}, {}
            random.seed(7)
            pc, ppc = ds.add_data(["tileP.txt"], 1)
            nc, npc = ds.add_data(["tileN.txt"], 0)
        finally:
            os.chdir(cwd)
    data = ds.data
    np.savez(os.path.join(OUT, "pair_sampler.npz"), fields=np.array(fields), pos_pairs=pos_pairs, neg_pairs=neg_pairs,
             seed=7, counts=np.array([pc, ppc, nc, npc]),
             out_tile=np.array([d[0] for d in data]), out_left=np.array([int(d[1]) for d in data]),
             out_right=np.array([int(d[2]) for d in data]), out_flag=np.array([d[3] for d in data]))


DESIGNED = ("area", "peri", "len", "width", "smooth", "std0", "std1", "std2", "mean0", "mean1", "mean2", "shapeness",
            "compact", "bright", "border")


def golden_pair_dataset(ref, rng):
    """The whole MergingSegmensPairDataset (MyUtils1.py:20-58, :236-295): add_data for a positive and a negative pair
    list over fake OGR / GDAL objects, then __getitem__ -> (left_meta, right_meta, flag) with
    meta = (designed [1,19], scales [1,4], [4 patches])."""
    R, H, W = 12, 90, 110
    arr = rng.integers(0, 256, size=(3, H, W)).astype(np.uint8)
    gt = (500.0, 2.0, 0.0, 1300.0, 0.0, -2.0)
    npts = rng.integers(1, 4, size=R)
    fields, pos = [], 0
    for r in range(R):
        fields.append(" ".join(str(pos + k) for k in range(npts[r])))
        pos += int(npts[r])
    N = pos
    attr = np.round(rng.uniform(0.5, 300.0, size=(N, 15)), 3)
    inner = rng.integers(6, 20, size=N)
    obj = inner + rng.integers(3, 25, size=N)
    X = gt[0] + rng.uniform(0, W - 1, size=N) * gt[1]
    Y = gt[3] + rng.uniform(0, H - 1, size=N) * gt[5]
    X[0], Y[0] = gt[0], gt[3]                                              # a corner point: zero-padded windows
    X[1], Y[1] = gt[0] + (W - 1) * gt[1], gt[3] + (H - 1) * gt[5]

    def point(i):
        f = dict(zip(DESIGNED, attr[i].tolist()))
        f["inner"], f["object"] = int(inner[i]), int(obj[i])
        return ref_shim.FakeFeature(i, f, (float(X[i]), float(Y[i])))

    polys = ref_shim.FakeLayer([ref_shim.FakeFeature(r, {"PointID": fields[r]}) for r in range(R)])
    pts = ref_shim.FakeLayer([point(i) for i in range(N)])
    pos_pairs = rng.integers(0, R, size=(9, 2))
    neg_pairs = rng.integers(0, R, size=(7, 2))
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            for name, pairs in (("tileA.txt", pos_pairs), ("tileB.txt", neg_pairs)):
                with open(name, "w") as f:
                    for j, (a, b) in enumerate(pairs):
                        f.write(f"{j},{a},{b},0,0\n")
            layers, rasters = {}, {}
            for t in ("tileA", "tileB"):
                layers[f"PF\\{t}.shp"] = polys
                layers[f"QF\\{t}\\PointsGCS.shp"] = pts
                rasters[f"IF\\{t}.tif"] = ref_shim.FakeRaster(arr, geotransform=gt)
            ref_shim.install_fake_drivers(ref, layers, rasters)
            ds = object.__new__(ref.MyUtils1.MergingSegmensPairDataset)
            ds.image_folder, ds.polygon_folder, ds.point_folder = "IF", "PF", "QF"
            ds.data, ds.point_dataset, ds.img_dataset, ds.layers = [], [], {}, {}
            random.seed(11)
            ds.positive_number, ds.positive_pair_number = ds.add_data(["tileA.txt"], 1)
            ds.negative_number, ds.negative_pair_number = ds.add_data(["tileB.txt"], 0)
        finally:
            os.chdir(cwd)
    out = {}
    for i in range(len(ds)):
        left, right, flag = ds[i]
        for side, meta in (("l", left), ("r", right)):
            out[f"{side}{i}_designed"] = meta[0].numpy()
            out[f"{side}{i}_scales"] = meta[1].numpy()
            for k, patch in enumerate(meta[2]):
                out[f"{side}{i}_patch{k}"] = patch
        out[f"flag{i}"] = np.int64(flag)
    golden.save(os.path.join(OUT, "pair_dataset.npz"), compressed=True, arr=arr, gt=np.array(gt), fields=np.array(fields), attr=attr,
                        inner=inner, obj=obj, X=X, Y=Y, pos_pairs=pos_pairs, neg_pairs=neg_pairs, seed=11, n=len(ds),
                        counts=np.array([ds.positive_number, ds.positive_pair_number, ds.negative_number,
                                         ds.negative_pair_number]),
                        data=np.array([[d[0], d[1], d[2], str(d[3])] for d in ds.data]), **out)


def golden_geometry(ref, rng):
    """calculate_left_top_point_and_size :379-383, get_scales :300-327, cut_image :330-360,
    pixel mapping :241-242 of MyUtils2.ExtractFeatureDataset."""
    ds = object.__new__(ref.MyUtils2.ExtractFeatureDataset)
    arr = rng.integers(0, 256, size=(3, 40, 50)).astype(np.uint8)
    ras = ref_shim.FakeRaster(arr, geotransform=(100.0, 0.5, 0.0, 900.0, 0.0, -0.5))
    ds.band_num = 3
    mids = np.array([[0, 0, 7], [3, 5, 8], [25, 20, 16], [49, 39, 9], [48, 2, 31], [10, 38, 12], [25, 20, 1]])
    wins = np.array([ds.calculate_left_top_point_and_size(int(x), int(y), int(w)) for x, y, w in mids])
    cuts = {f"cut{i}": ds.cut_image(ras, tuple(int(v) for v in wins[i])) for i in range(len(mids))}
    io = np.array([[8, 20], [15, 15], [30, 70], [5, 6]])
    sc = [ds.get_scales(int(a), int(b)) for a, b in io]
    geo = np.array([[100.0, 900.0], [103.3, 893.2], [124.4, 880.6], [112.25, 899.75]])
    gt = ras.GetGeoTransform()
    px = np.array([[int(abs((gt[0] - x) / gt[1]) + 1), int(abs((gt[3] - y) / gt[5]) + 1)] for x, y in geo])
    np.savez(os.path.join(OUT, "geometry.npz"), arr=arr, gt=np.array(gt), mids=mids, wins=wins, io=io,
             scales=np.array([s[0] for s in sc]), factors=np.array([s[1] for s in sc]),
             cfg_scales=np.array(ref.config.configs.scales), geo=geo, px=px, **cuts)


def golden_resize(ref, rng):
    """ExtractFeatureDataset.resize_data :362-376 (cv2.resize INTER_AREA per band, then / 255) on the patch sizes the
    loader meets: integer shrink factors 1, 2, 3, 4, fractional shrinks, enlargements, the 1 x 1 environment patch."""
    ds = object.__new__(ref.MyUtils2.ExtractFeatureDataset)
    cases = [(32, 32), (64, 32), (96, 32), (128, 32), (50, 32), (45, 32), (20, 32), (31, 32), (128, 64), (90, 64),
             (70, 64), (40, 64), (200, 128), (129, 128), (100, 128), (64, 128), (37, 1), (64, 1), (150, 1)]
    out = {}
    for i, (s_, t) in enumerate(cases):
        ds.band_num = 3 if i == 4 else 1                                       # (small fixtures: one band mostly)
        patch = rng.integers(0, 256, size=(ds.band_num, s_, s_)).astype(np.uint8)
        if i % 3 == 0:
            patch[:, : s_ // 3] = 0                                            # zero padding of a border window
        out[f"in{i}"] = patch
        out[f"out{i}"] = ds.resize_data(patch, t, t)
    np.savez_compressed(os.path.join(OUT, "resize.npz"), cases=np.array(cases), **out)


def main():
    if not ref_shim.available():
        raise SystemExit("needs /root/reference (build container only)")
    os.makedirs(OUT, exist_ok=True)
    ref = ref_shim.load()
    only = set(sys.argv[1:])                          # optional: names of the generators to run
    rng = np.random.default_rng(20261018)
    for fn in (golden_euclid, golden_pool_score, golden_mlp, golden_loss, golden_edge_reader,
               golden_pair_sampler, golden_geometry, golden_resize):
        if only and fn.__name__ not in only:
            # keep the shared random stream in step: run the generator into a scratch directory
            continue
        fn(ref, rng)
        print("wrote", fn.__name__)
    # generators added later draw from streams of their own, so that the fixtures above never change
    for fn, seed in ((golden_pair_dataset, 20261019),):
        if only and fn.__name__ not in only:
            continue
        fn(ref, np.random.default_rng(seed))
        print("wrote", fn.__name__)


if __name__ == "__main__":
    main()
