"""Times deepmerge_b200.rasterize on the configs[1] scene (10k x 10k, ~100k segments; not part of the merge step): the
unmerged synthetic labels and the merged label map of MergeEngine.run, each polygonized on the GPU, with the flat rings
(float64 pixel-corner vertices, one record per region, identity geotransform) resident on the device.  Prints one JSON
line with ms (CUDA events over the calls after 3 warm-up calls, the whole call including its read-back of the counts),
the crossings, spans and pixels painted, the algorithmic bytes 16 n_vertices + 12 crossings + 4 H W and their rate
against the 7.7 TB/s HBM data sheet figure, and, on the same map written with write_polygonized, the host time of
shapefile.read_polygon_rings, read_polygons and rasterize_polygons, and the card's name and power limit.  Every result
is checked against the map it came from.

    python tools/time_rasterize.py [--calls 20]
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from deepmerge_b200 import MergeEngine, _lib, polygonize, rasterize, synth  # noqa: E402
from deepmerge_b200 import shapefile as shp  # noqa: E402
from time_polygonize import DATASHEET_HBM_GBS, card  # noqa: E402

IDENTITY = (0.0, 1.0, 0.0, 0.0, 0.0, 1.0)


def counts_of(rings, H, W):
    """counts of dm_rasterize at the exact capacity (a first call at capacity 0 finds it): spans, pixels, crossings,
    status."""
    L = _lib.lib()
    xy, off, rec, n = rings
    out = torch.empty((H, W), dtype=torch.int32, device=xy.device)

    def call(cap):
        counts = torch.zeros(4, dtype=torch.int64, device=xy.device)
        ws_bytes = L.dm_rasterize_workspace_bytes(xy.shape[0], n, cap)
        ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=xy.device)
        L.check(L.dm_rasterize(xy.data_ptr(), xy.shape[0], off.data_ptr(), rec.data_ptr(), rec.shape[0], n, 0.0, 1.0, 0.0,
                               1.0, None, -1, H, W, W, cap, out.data_ptr(), counts.data_ptr(), ws.data_ptr(), ws_bytes,
                               torch.cuda.current_stream().cuda_stream), "dm_rasterize")
        return counts.tolist()

    c = call(call(0)[2])
    assert c[3] == 0, c
    return c


def time_one(labels, R, calls, tmp):
    H, W = labels.shape
    P = polygonize(labels, R)
    rings = shp.PolygonRings(P.vertices.double().contiguous(), P.ring_offsets, P.ring_region, R)
    for _ in range(3):
        out = rasterize(rings, IDENTITY, H, W)
    assert torch.equal(out, labels)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        out = rasterize(rings, IDENTITY, H, W)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / calls
    spans, pixels, crossings, _ = counts_of(rings, H, W)
    n_v = int(rings.xy.shape[0])
    nbytes = 16 * n_v + 12 * crossings + 4 * H * W
    # the host path on the same polygons, through a file
    path = os.path.join(tmp, "tile.shp")
    shp.write_polygonized(path, P, IDENTITY)
    t0 = time.perf_counter()
    flat = shp.read_polygon_rings(path)
    t1 = time.perf_counter()
    polys = shp.read_polygons(path)
    t2 = time.perf_counter()
    ids = shp.DbfTable(path[:-4] + ".dbf").column_int("REGION")
    t3 = time.perf_counter()
    host = shp.rasterize_polygons(polys, IDENTITY, H, W, ids=ids)
    t4 = time.perf_counter()
    assert np.array_equal(host, labels.cpu().numpy())
    assert torch.equal(rasterize(flat, IDENTITY, H, W, ids=ids), labels)
    return {"ms": round(ms, 3), "polygons": int(P.region_rings.diff().gt(0).sum()), "rings": P.n_rings, "vertices": n_v,
            "crossings": crossings, "spans": spans, "pixels_painted": pixels, "alg_bytes": nbytes,
            "gbs": round(nbytes / ms / 1e6, 1), "frac_hbm_datasheet": round(nbytes / ms / 1e6 / DATASHEET_HBM_GBS, 4),
            "host_read_polygon_rings_s": round(t1 - t0, 3), "host_read_polygons_s": round(t2 - t1, 3),
            "host_rasterize_polygons_s": round(t4 - t3, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=20)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    sc = synth.synth_scene(10000, 10000, 100000, C=4, device=dev)
    eng = MergeEngine(10000, 10000, sc.n_regions, sc.feats.shape[1], C=4, n_points=sc.feats.shape[0], device=dev)
    res = eng.run(sc.labels, sc.feats, 0.5, image=sc.image, xs=sc.xs, ys=sc.ys)
    merged = res.labels.clone()
    name, power = card()
    out = {"tool": "time_rasterize", "scene": "configs[1] 10k x 10k, %d regions" % sc.n_regions, "card": name,
           "power_limit": power, "calls": args.calls, "hbm_datasheet_gbs": DATASHEET_HBM_GBS}
    with tempfile.TemporaryDirectory() as tmp:
        out["unmerged"] = time_one(sc.labels, sc.n_regions, args.calls, tmp)
        out["merged"] = dict(time_one(merged, sc.n_regions, args.calls, tmp), regions_left=sc.n_regions - res.merges)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
