"""Times polygonize and boundary_lines with a tolerance (dm_polygonize_simplified / dm_lines_simplified; not part of
the merge step) on the configs[1] scene (10k x 10k, ~100k segments), the merged label map of MergeEngine.run and the
unmerged synthetic labels, against the plain calls in the same run.  Each input is 400 MB of labels, more than the
126 MB L2, so every call reads it from HBM.  Prints one JSON line with ms per call (CUDA events over the calls after
warm-up, the whole call including its read-back of the counts) at t = 0.5, 1 and 2 px and without simplification, the
vertex counts before and after, the host time of the sequential simplifier of tests/simplify_oracle.c at t = 1 (its
tracing by the oracles of tests/polygon_oracle.c / lines_oracle.c excluded), and the card's name and power limit.

    python tools/time_simplify.py [--calls 20]
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
from deepmerge_b200 import MergeEngine, boundary_lines, polygonize, synth  # noqa: E402
import lines_oracle as lo  # noqa: E402  (the sequential tracers and simplifier the tests compare against)
import polygon_oracle as po  # noqa: E402
import simplify_oracle as so  # noqa: E402
from time_polygonize import card  # noqa: E402

TOLERANCES = (0.5, 1.0, 2.0)


def ms_per_call(fn, calls):
    for _ in range(3):
        out = fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return round(a.elapsed_time(b) / calls, 3), out


def time_map(labels, R, calls):
    out = {}
    for name, f in (("polygonize", polygonize), ("boundary_lines", boundary_lines)):
        row = {}
        ms, P = ms_per_call(lambda: f(labels, R), calls)
        row["plain"] = {"ms": ms, "vertices": int(P.vertices.shape[0])}
        for t in TOLERANCES:
            ms, P = ms_per_call(lambda: f(labels, R, tolerance=t), calls)
            row["t=%g" % t] = {"ms": ms, "vertices": int(P.vertices.shape[0])}
        out[name] = row
    L = labels.cpu().numpy()
    H, W = L.shape
    P = po.polygonize(L, R)
    v, off, node = so.ring_nodes(L, P)
    out["polygonize"]["vertices_with_nodes"] = int(len(v))
    t0 = time.perf_counter()
    so.keep(v, off, H, W, 1.0, node)
    out["polygonize"]["oracle_simplify_host_s_t1"] = round(time.perf_counter() - t0, 3)
    Q = lo.lines(L, R)
    t0 = time.perf_counter()
    so.keep(Q["vertices"], Q["line_offsets"], H, W, 1.0)
    out["boundary_lines"]["oracle_simplify_host_s_t1"] = round(time.perf_counter() - t0, 3)
    return out


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
    out = {"tool": "time_simplify", "scene": "configs[1] 10k x 10k, %d regions" % sc.n_regions, "card": name,
           "power_limit": power, "calls": args.calls}
    for key, labels in (("merged", merged), ("unmerged", sc.labels)):
        out[key] = time_map(labels, sc.n_regions, args.calls)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
