"""Dev check: pipelined host path vs device path, report differing cells (GPU)."""
import os, sys
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools']
import torch, bench
import traversability_estimation_b200 as te
rows, cols = 2048, 2304
z = bench.terrain_torch(torch, rows, 0, cols, cols, 9, 0.01, torch.device("cuda"))
g, p = te.Geometry.make(rows, cols, 0.02), te.ChainParams.yaml_defaults(0)
ctx = te.Context(0)
if len(sys.argv) > 1:   # what test_size_independent_properties_at_scale does before, in the same context
    r4 = 4096
    z4 = bench.terrain_torch(torch, r4, 0, r4, r4, 7, 0.01, torch.device("cuda"))
    g4 = te.Geometry.make(r4, r4, 0.02)
    a = [torch.empty((r4, r4), dtype=torch.float32, device="cuda") for _ in range(4)]
    b = [torch.empty((r4, r4), dtype=torch.float32, device="cuda") for _ in range(4)]
    ctx.chain(g4, p, z4, *a, te.MEM_DEVICE)
    ctx.chain(g4, p, z4, *b, te.MEM_DEVICE)
    ctx.synchronize()
    print("4096 pair equal:", [bool(torch.equal(x.view(torch.int32), y.view(torch.int32))) for x, y in zip(a, b)])
    g5 = te.Geometry.make(r4, r4, 0.02, (123.456, -78.9))
    ctx.chain(g5, p, z4, *b, te.MEM_DEVICE)
    ctx.synchronize()
dev = [torch.empty((cols, rows), dtype=torch.float32, device="cuda") for _ in range(4)]
ctx.chain(g, p, z, *dev, te.MEM_DEVICE)
ctx.synchronize()
print("device flags", ctx.flag_counters())
h_in = z.cpu().pin_memory()
h_out = [torch.empty((cols, rows), dtype=torch.float32).pin_memory() for _ in range(4)]
ctx.chain(g, p, h_in.data_ptr(), *[o.data_ptr() for o in h_out], te.MEM_HOST)
for name, a, b in zip(("slope", "step", "rough", "trav"), dev, h_out):
    a = a.cpu()
    d = (a.view(torch.int32) != b.view(torch.int32))
    n = int(d.sum())
    print(name, "differs in", n)
    if n:
        idx = d.nonzero()
        print("  columns", int(idx[:, 0].min()), int(idx[:, 0].max()), "rows", int(idx[:, 1].min()), int(idx[:, 1].max()))
        print("  first", [(int(j), int(i), float(a[j, i]), float(b[j, i])) for j, i in idx[:8]])
        cols_hist = torch.bincount(idx[:, 0] // 128, minlength=18)
        print("  per 128-col block", cols_hist.tolist())
