"""Time the edge sort / sort+unique primitives alone (CUDA events): tools/prof_sort.py [n [R [reps]]]."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from deepmerge_b200 import _lib

n = int(sys.argv[1]) if len(sys.argv) > 1 else 650000
R = int(sys.argv[2]) if len(sys.argv) > 2 else 98000
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
L = _lib.lib()
dev = torch.device("cuda:0")
rng = np.random.default_rng(1)
lo = rng.integers(0, R, n)
hi = np.minimum(R - 1, lo + rng.integers(0, 40, n))          # ~ a region graph: many duplicates
keys0 = torch.from_numpy(((lo.astype(np.uint64) << np.uint64(32)) | hi.astype(np.uint64)).view(np.int64)).to(dev)
vals0 = torch.ones(n, dtype=torch.int32, device=dev)
cap = n + 1000
k = torch.empty(cap, dtype=torch.int64, device=dev)
v = torch.empty(cap, dtype=torch.int32, device=dev)
nd = torch.tensor([n], dtype=torch.int64, device=dev)
nout = torch.zeros(1, dtype=torch.int64, device=dev)
wsb = max(L.dm_sort_edges_workspace_bytes(cap), L.dm_edges_unique_workspace_bytes(cap))
ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
s = torch.cuda.current_stream().cuda_stream


def timed(fn):
    ms = []
    for _ in range(reps):
        k[:n].copy_(keys0)
        v[:n].copy_(vals0)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    return sorted(ms)[len(ms) // 2] * 1000


t_sort = timed(lambda: L.check(L.dm_sort_edges(k.data_ptr(), v.data_ptr(), nd.data_ptr(), cap, R, ws.data_ptr(), wsb, s), "sort"))
t_uniq = timed(lambda: L.check(L.dm_edges_sort_unique(k.data_ptr(), v.data_ptr(), nd.data_ptr(), cap, R, nout.data_ptr(),
                                                       ws.data_ptr(), wsb, s), "sort_unique"))
print("n=%d R=%d: sort %.1f us, sort+unique %.1f us (%d unique)" % (n, R, t_sort, t_uniq, int(nout.item())))
