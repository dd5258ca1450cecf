"""Times deepmerge_b200.polygonize on the configs[1] scene (10k x 10k, ~100k segments; not part of the merge step):
the merged label map of MergeEngine.run and the unmerged synthetic labels.  Each input is 400 MB of labels, more than
the 126 MB L2, so every call reads it from HBM.  Prints one JSON line with ms (CUDA events over the calls after
warm-up, the whole call including its read-back of the counts), the sides / rings / vertices found, the algorithmic
bytes 4 H W + 8 n_vertices + 20 n_rings + 8 n_regions and their rate against the HBM peak, the host time of the
sequential C tracer of tests/polygon_oracle.c on the same map, and the card's name and power limit.

    python tools/time_polygonize.py [--calls 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from deepmerge_b200 import MergeEngine, polygonize, synth  # noqa: E402
import polygon_oracle as po  # noqa: E402  (the sequential tracer the tests compare against)

DATASHEET_HBM_GBS = 7700.0


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except (OSError, KeyError, ValueError):
        return DATASHEET_HBM_GBS, "data sheet"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def time_one(labels, R, calls):
    for _ in range(3):
        P = polygonize(labels, R)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        P = polygonize(labels, R)
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / calls
    H, W = labels.shape
    nbytes = 4 * H * W + 8 * P.vertices.shape[0] + 20 * P.n_rings + 8 * R
    L = labels.cpu().numpy()
    t0 = time.perf_counter()
    po.polygonize(L, R)
    host_s = time.perf_counter() - t0
    peak, src = hbm_peak()
    return {"ms": round(ms, 3), "boundary_sides": P.boundary_sides, "rings": P.n_rings, "vertices": int(P.vertices.shape[0]),
            "alg_bytes": nbytes, "gbs": round(nbytes / ms / 1e6, 1), "frac_hbm_peak": round(nbytes / ms / 1e6 / peak, 4),
            "hbm_peak_gbs": peak, "hbm_peak_source": src, "oracle_host_s": round(host_s, 3)}


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
    out = {"tool": "time_polygonize", "scene": "configs[1] 10k x 10k, %d regions" % sc.n_regions, "card": name,
           "power_limit": power, "calls": args.calls,
           "merged": dict(time_one(merged, sc.n_regions, args.calls), regions_left=sc.n_regions - res.merges),
           "unmerged": time_one(sc.labels, sc.n_regions, args.calls)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
