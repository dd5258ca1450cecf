"""Times deepmerge_b200.boundary_lines on the configs[1] scene (10k x 10k, ~100k segments; not part of the merge step),
the merged label map of MergeEngine.run and the unmerged synthetic labels, with polygonize on the same maps in the same
run.  Each input is 400 MB of labels, more than the 126 MB L2, so every call reads it from HBM.  Prints one JSON line
with ms (CUDA events over the calls after warm-up, the whole call including its read-back of the counts), the
segments / lines / vertices found, the algorithmic bytes 4 H W + 8 n_vertices + 24 n_lines and their rate against the
HBM peak, the host time of the sequential C tracer of tests/lines_oracle.c on the same map, polygonize's line of
tools/time_polygonize.py, and the card's name and power limit.

    python tools/time_lines.py [--calls 20]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
from deepmerge_b200 import MergeEngine, boundary_lines, synth  # noqa: E402
import lines_oracle as lo  # noqa: E402  (the sequential tracer the tests compare against)
from time_polygonize import card, hbm_peak, time_one as time_polygonize  # noqa: E402


def time_one(labels, R, calls):
    for _ in range(3):
        P = boundary_lines(labels, R)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        P = boundary_lines(labels, R)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / calls
    H, W = labels.shape
    nbytes = 4 * H * W + 8 * P.vertices.shape[0] + 24 * P.n_lines
    L = labels.cpu().numpy()
    t0 = time.perf_counter()
    lo.lines(L, R)
    host_s = time.perf_counter() - t0
    peak, src = hbm_peak()
    return {"ms": round(ms, 3), "boundary_segments": P.boundary_segments, "lines": P.n_lines,
            "vertices": int(P.vertices.shape[0]), "alg_bytes": nbytes, "gbs": round(nbytes / ms / 1e6, 1),
            "frac_hbm_peak": round(nbytes / ms / 1e6 / peak, 4), "hbm_peak_gbs": peak, "hbm_peak_source": src,
            "oracle_host_s": round(host_s, 3)}


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
    out = {"tool": "time_lines", "scene": "configs[1] 10k x 10k, %d regions" % sc.n_regions, "card": name,
           "power_limit": power, "calls": args.calls}
    for key, labels in (("merged", merged), ("unmerged", sc.labels)):
        out[key] = time_one(labels, sc.n_regions, args.calls)
        out[key]["polygonize_ms"] = time_polygonize(labels, sc.n_regions, args.calls)["ms"]
    out["merged"]["regions_left"] = sc.n_regions - res.merges
    print(json.dumps(out))


if __name__ == "__main__":
    main()
