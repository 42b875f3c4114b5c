import os, sys
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools', _R + '/tests']
import numpy as np, synth
import traversability_estimation_b200 as te
ctx = te.Context(0)
for (rows, cols, res) in [(128, 96, 0.02), (64, 250, 0.02), (100, 60, 0.03)]:
    z = synth.terrain(rows, cols, res, 3, 'mixed')
    g = te.Geometry.make(rows, cols, res)
    ctx.set_kernel(te.KERNEL_AUTO)
    o = ctx.chain_host(g, te.ChainParams.yaml_defaults(0), z)
    fp = te.FootprintParams.yaml_defaults()
    out = np.empty((rows, cols), np.float32, order='F')
    t, s, st = (np.asfortranarray(o[k]) for k in ('traversability', 'slope', 'step'))
    ctx.footprint(g, fp, t, s, st, np.asfortranarray(z), out, te.MEM_HOST)
    print(rows, cols, np.nanmean(o['traversability']), np.nanmean(out))
ctx.close()
