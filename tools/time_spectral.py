"""Times MergeEngine.run_spectral (merge by spectral and shape heterogeneity, no embeddings) on the configs[1] scene
(10k x 10k, 4 bands, ~98k regions) at scale 60, shape 0.1, compactness 0.5.  Prints one JSON line: the card's name and
power limit; rounds and regions left; ms per whole call (CUDA events over the calls after warm-up: raster pass, boxes,
every round and the relabel) and per round; and the score kernel timed alone on the initial graph (every edge scored,
CUDA events over many launches) with its algorithmic bytes -- per edge its key, length and score, per endpoint area,
perimeter, box and the C band sums and sums of squares, 2 (40 + 16 C) + 16 bytes -- and their rate against the HBM
peak.  The gathered rows (~12 MB) fit the 126 MB L2, so the rate is an effective one, not an HBM measurement.

    python tools/time_spectral.py [--calls 10]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from deepmerge_b200 import MergeEngine, _lib, build_rag, synth  # noqa: E402
from time_polygonize import card, hbm_peak  # noqa: E402

SCALE, SHAPE, CMPCT = 60.0, 0.1, 0.5


def events(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=10)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    sc = synth.synth_scene(10000, 10000, 100000, C=4, device=dev, with_image=True)
    R, C = sc.n_regions, 4
    eng = MergeEngine(10000, 10000, R, 0, C=C, n_points=0, device=dev)
    run = lambda: eng.run_spectral(sc.labels, sc.image, SCALE, shape=SHAPE, compactness=CMPCT)
    for _ in range(2):
        res = run()
    ms = events(run, args.calls)
    rounds, left = res.rounds, R - res.merges

    rag = build_rag(sc.labels, R, sc.image, bbox=True)
    E = rag.n_edges
    L = _lib.lib()
    n = torch.tensor([E], dtype=torch.int64, device=dev)
    scores = torch.empty(E, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream().cuda_stream
    score = lambda: L.check(L.dm_score_spectral(rag.edge_keys.data_ptr(), rag.boundary_len.data_ptr(), n.data_ptr(), E,
                                                rag.area.data_ptr(), rag.perimeter.data_ptr(), rag.band_sum.data_ptr(),
                                                rag.band_sumsq.data_ptr(), C, rag.bbox.data_ptr(), None, SHAPE, CMPCT, None,
                                                scores.data_ptr(), s), "dm_score_spectral")
    events(score, 20)
    score_ms = events(score, 200)
    nbytes = E * (2 * (40 + 16 * C) + 16)
    peak, src = hbm_peak()
    out = {"tool": "time_spectral", "scene": "configs[1] 10k x 10k, %d regions, C = %d" % (R, C), "card": card()[0],
           "power_limit": card()[1], "scale": SCALE, "shape": SHAPE, "compactness": CMPCT, "calls": args.calls,
           "rounds": rounds, "regions_left": left, "ms_per_call": round(ms, 3),
           "ms_per_round": round(ms / max(rounds, 1), 3),
           "score_kernel": {"edges": E, "ms": round(score_ms, 4), "alg_bytes": nbytes,
                            "gbs": round(nbytes / score_ms / 1e6, 1),
                            "frac_hbm_peak": round(nbytes / score_ms / 1e6 / peak, 4), "hbm_peak_gbs": peak,
                            "hbm_peak_source": src}}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
