"""Run only the fused RAG + band-pooling raster pass a few times (ncu / timing target)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from deepmerge_b200 import MergeEngine, _lib
from deepmerge_b200.raster import _p, _stream
from deepmerge_b200.synth import synth_scene

side = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
R = int(sys.argv[2]) if len(sys.argv) > 2 else int(100000 * side * side / 1e8)
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 3
C = int(sys.argv[4]) if len(sys.argv) > 4 else 4
if os.environ.get('DM_LIB'):
    _lib._LIB = _lib.Library(os.environ['DM_LIB'])
L = _lib.lib()
dev = torch.device("cuda:0")
sc = synth_scene(side, side, R, C=C, device=dev)
eng = MergeEngine(side, side, sc.n_regions, 100, C=C, n_points=sc.feats.shape[0], device=dev)
ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
for a, b in ev:
    eng.stats.zero_()
    a.record()
    L.check(L.dm_rag_scan(_p(sc.labels), side, side, side, side, _p(sc.image), C, side * C, sc.n_regions, 1, 1, _p(eng.area),
                          _p(eng.border), _p(eng.bsum), _p(eng.bsq), eng.cap, _p(eng.counts), _p(eng.ws), eng.ws_bytes,
                          _stream()), "scan")
    b.record()
torch.cuda.synchronize()
ms = [a.elapsed_time(b) for a, b in ev]
byts = (4 + C) * side * side
print("path", L.dm_rag_last_path(), "encode_err", L.dm_rag_last_encode_error(), "counts", eng.counts.tolist()[:4])
print("ms", ms, "GB/s", [byts / m / 1e6 for m in ms])
