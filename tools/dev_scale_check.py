"""One-off: fused vs literal kernel on the bench map itself (8192 x 8192, 1 % holes)."""
import os, sys
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools']
import torch, bench
import traversability_estimation_b200 as te
rows = cols = 8192
z = bench.terrain_torch(torch, rows, 0, cols, cols, 3, 0.01, torch.device('cuda'))
g = te.Geometry.make(rows, cols, 0.02); p = te.ChainParams.yaml_defaults(0)
ctx = te.Context(0); res = {}
for name, k in (('fused', te.KERNEL_FUSED), ('literal', te.KERNEL_GENERIC)):
    ctx.set_kernel(k)
    outs = [torch.empty((cols, rows), dtype=torch.float32, device='cuda') for _ in range(4)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.chain(g, p, z, *outs, te.MEM_DEVICE); ctx.synchronize()
    ctx.enable_timing(True); ctx.chain(g, p, z, *outs, te.MEM_DEVICE); print(name, 'ms', ctx.timing()); ctx.enable_timing(False)
    res[name] = outs
for kname, a, b in zip(('slope', 'step', 'roughness', 'traversability'), res['fused'], res['literal']):
    nanmis = int((torch.isnan(a) != torch.isnan(b)).sum())
    ok = ~torch.isnan(b) & ~torch.isnan(a)
    d = (a[ok].double() - b[ok].double()).abs(); tol = 1e-5 * b[ok].double().abs() + 1e-6
    print(kname, 'nan mismatches', nanmis, 'out of tol', int((d > tol).sum()), 'worst err/tol', float((d / tol).max()),
          'bit-exact', float((a[ok] == b[ok]).double().mean()))
print('flag counters', ctx.flag_counters())
