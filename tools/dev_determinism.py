"""Dev check: run the fused chain twice on the same map and report cells whose bits differ (GPU)."""
import os, sys
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools']
import torch, bench
import traversability_estimation_b200 as te
rows = cols = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
z = bench.terrain_torch(torch, rows, 0, cols, cols, 7, 0.01, torch.device("cuda"))
g, p = te.Geometry.make(rows, cols, 0.02), te.ChainParams.yaml_defaults(0)
ctx = te.Context(0)
runs = []
b2b = len(sys.argv) > 2
for r in range(6):
    o = [torch.empty((cols, rows), dtype=torch.float32, device="cuda") for _ in range(4)]
    ctx.chain(g, p, z, *o, te.MEM_DEVICE)
    if not b2b:
        ctx.synchronize()
        print("run", r, "flags", ctx.flag_counters())
    runs.append(o)
ctx.synchronize()
for r in (1, 2, 3, 4, 5):
    for name, a, b in zip(("slope", "step", "rough", "trav"), runs[0], runs[r]):
        d = (a.view(torch.int32) != b.view(torch.int32))
        n = int(d.sum())
        if n:
            idx = d.nonzero()[:5]
            print("run", r, name, "differs in", n, "cells; first", [(int(j), int(i), float(a[j, i]), float(b[j, i])) for j, i in idx])
print("done")
