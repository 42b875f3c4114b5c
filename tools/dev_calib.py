"""Calibration run: flagged-cell count and fp32 error against the oracle for a sweep of the certification constants (dev tool, GPU).

Needs a calibration build, which is the only one that reads TE_FUSED_ROUGH_K / TE_FUSED_COND_K:
    make -C traversability_estimation_b200/csrc variant NAME=calib EXTRA=-DTE_CALIBRATION=1
    TE_B200_LIBRARY=$PWD/traversability_estimation_b200/libte_b200_calib.so python tools/dev_calib.py
"""
import os, sys, json
_R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path[:0] = [_R, _R + '/tools', _R + '/tests']
import numpy as np, synth, torch, bench
import traversability_estimation_b200 as te
from oracle import binding as ob
from helpers import compare_layer
rows = cols = 1024
dev = torch.device('cuda', 0)
z_t = bench.terrain_torch(torch, rows, 0, cols, cols, 3, 0.0, dev)
z = np.asfortranarray(z_t.cpu().numpy().T)
og = ob.Geometry.make(rows, cols, 0.02); g = te.Geometry.make(rows, cols, 0.02)
ref = ob.chain(og, ob.ChainParams.yaml_defaults(0), z)
for rk, ck in [(0.2, 0.25), (0.1, 0.25), (0.05, 0.25), (0.0, 0.25), (0.1, 0.1), (0.1, 0.0), (0.05, 0.1)]:
    os.environ['TE_FUSED_ROUGH_K'] = str(rk); os.environ['TE_FUSED_COND_K'] = str(ck)
    ctx = te.Context(0); ctx.set_kernel(te.KERNEL_FUSED)
    got = ctx.chain_host(g, te.ChainParams.yaml_defaults(0), z)
    cnt = ctx.flag_counters()
    rep = {k: compare_layer(got[k], ref[k], k) for k in ('slope', 'roughness', 'traversability')}
    print(f"rough_k={rk} cond_k={ck} flagged={cnt} frac={cnt[0]/rows/cols:.4f}  " +
          "  ".join(f"{k}: oot={r['out_of_tol']} max={r['max_abs']:.2e}" for k, r in rep.items()))
    ctx.close()
