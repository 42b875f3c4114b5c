import os, sys, time
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools', _R + '/tests']
import numpy as np, synth
import traversability_estimation_b200 as te
from oracle import binding as ob
from helpers import compare_layer
ctx = te.Context(0)
for (rows, cols, seed, preset, res) in [(128, 96, 1, 'gentle', 0.02), (256, 200, 2, 'mixed', 0.02), (512, 384, 3, 'rough', 0.02), (1024, 768, 4, 'mixed', 0.02), (200, 160, 5, 'mixed', 0.03)]:
    z = synth.terrain(rows, cols, res, seed, preset)
    g = te.Geometry.make(rows, cols, res); og = ob.Geometry.make(rows, cols, res)
    ref = ob.chain(og, ob.ChainParams.yaml_defaults(0), z, with_normals=True)
    ctx.set_kernel(te.KERNEL_FUSED)
    got = ctx.chain_host(g, te.ChainParams.yaml_defaults(0), z, with_normals=True)
    cnt = ctx.flag_counters()
    print(rows, cols, preset, res, 'tier2 cells', cnt[0], 'tier3 cells', cnt[4], 'of', rows*cols)
    for k in ('slope','step','roughness','traversability','nx','ny','nz'):
        r = compare_layer(got[k], ref[k], k)
        print('   ', {kk: r[kk] for kk in ('name','nan_mismatch','out_of_tol','rel_only_violations','branch_mismatch','bit_exact','max_abs')})
