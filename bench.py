#!/usr/bin/env python
"""bench.py — Mcells/s of the full filter chain on synthetic elevation (BASELINE.json metric).

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU restatement of the reference chain (oracle) on host cores

A "step" is one pass of the hot path (elevation -> slope, step, roughness, traversability) over one
map: the 8192 x 8192 map of BASELINE config 3, the one the >=70 %-of-roofline target is quoted on.  At N>1
the SAME map is tiled into N column slabs (strong scaling, config 3 verbatim): every rank owns 8192 rows x
8192/N columns and pulls the 4 boundary columns of `elevation` of each neighbour into its halo inside
the step — by default straight out of the neighbour's buffer over NVLink (CUDA IPC mapping, te_halo_pull
of the C ABI; `--halo nccl` uses NCCL send/recv instead).  `--scaling weak` grows the map with N instead
(every rank an 8192 x 8192 slab of an 8192 x 8192*N map).
torch is plumbing only (device memory, streams, torch.distributed); every kernel timed here is ours,
called through the C ABI of libte_b200.so.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

ALG_BYTES_PER_CELL = 20  # read elevation 4 B + write slope, step, roughness, traversability (SURVEY.md §8d)
RES = 0.02


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    # default: 400 (>= 0.2 s of timed device work at 8192^2); 20 for --impl reference and 5 for --workload plugin_chain,
    # whose steps take seconds (host CPU) and hundreds of milliseconds (host GridMaps, timed twice) each
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="chain8192", choices=["chain8192", "chain2048", "batched512", "footprint4096", "footprint4096_offset0", "footprint_polygon4096", "slope8192", "plugin_chain"])
    ap.add_argument("--scaling", default="strong", choices=["weak", "strong"])
    ap.add_argument("--halo", default="ipc", choices=["ipc", "nccl"], help="halo exchange at N>1: peer-mapped pull (C ABI) or NCCL send/recv")
    ap.add_argument("--halo-overlap", type=int, default=1, help="N>1, --halo ipc: pull the halo of the NEXT buffer set on a side stream while the chain runs on the current one (0: inline, on the chain's stream)")
    ap.add_argument("--kernel", default="auto", choices=["auto", "generic", "fused"])
    ap.add_argument("--holes", type=float, default=0.01, help="fraction of NaN cells (blobs)")
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the layers the last timed step computed as DIR/<name>.npy, their NaN "
                         "cells as DIR/<name>_nan.npy (see dump_outputs), so that two builds can be compared output for output; "
                         "--impl reference writes DIR/reference_<name>.npy for its top-left crop, comparable only with itself")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 5 if args.workload == "plugin_chain" else 400
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload == "plugin_chain":
        ap.error("--dump-outputs is not available for --workload plugin_chain: its timed passes run inside the C++ harness")
    return args


DUMP_BYTES = 60_000_000  # all .npy files of one --dump-outputs run together stay below 64 MB
DUMP_SEED = 7


def dump_outputs(path, arrays, dist=None, world=1, rank=0):
    """`--dump-outputs DIR`: write every array of `arrays` (name -> this rank's tensor or column-major numpy layer, all of one
    size) as DIR/<name>.npy, 1-D in the array's dtype.  The whole array is the ranks' shares concatenated in rank order and
    flattened in storage order (a column-major layer: index col * rows + row; a batch of maps: one map after the other), so
    that a run on N GPUs writes the same files as a run on one.  Arrays too large for their share of DUMP_BYTES are written
    at a sorted, seeded sample of flat indices, which depends only on the size: the same cells in every run and every build.
    Every written value is finite: a cell where a layer holds NaN (no data; the chain answers so for most cells whose input
    elevation is NaN) is written as 0.0 in <name>.npy and as 1.0 in DIR/<name>_nan.npy, which holds 0.0 at every other cell,
    so the two files carry the layer's values and its NaN pattern at every sampled cell.  Collective at N > 1 (every rank
    calls it); rank 0 writes."""
    import torch

    def flat(a):
        return a.reshape(-1) if torch.is_tensor(a) else torch.from_numpy(np.ravel(a, order="F"))

    arrays = {name: flat(a) for name, a in arrays.items()}
    first = next(iter(arrays.values()))
    dev, n_local = first.device, first.numel()
    assert all(a.numel() == n_local for a in arrays.values())
    n_total = n_local * world
    k = DUMP_BYTES // (2 * len(arrays)) // max(a.element_size() for a in arrays.values())   # values + NaN pattern
    if n_total <= k:
        idx = torch.arange(n_total, device=dev)
    else:
        idx = torch.from_numpy(np.unique(np.random.default_rng(DUMP_SEED).integers(0, n_total, k))).to(dev)
    owner = idx // n_local
    mine = owner == rank
    if rank == 0:
        os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        vals = torch.zeros((idx.numel(),), dtype=a.dtype, device=dev)
        vals[mine] = a.to(dev)[idx[mine] - rank * n_local]
        if world > 1:
            parts = [torch.empty_like(vals) for _ in range(world)]
            dist.all_gather(parts, vals)
            vals = torch.stack(parts)[owner, torch.arange(idx.numel(), device=dev)]
        if rank == 0:
            nan = torch.isnan(vals)
            np.save(os.path.join(path, name + ".npy"), torch.where(nan, torch.zeros_like(vals), vals).cpu().numpy())
            np.save(os.path.join(path, name + "_nan.npy"), nan.to(vals.dtype).cpu().numpy())


# ------------------------------------------------------------------------------------------------
# synthetic terrain, generated on the device as a pure function of GLOBAL cell coordinates so every
# rank can build its own slab (spectral fBm + mm noise + raised rectangles + flat patches + NaN blobs)
# ------------------------------------------------------------------------------------------------
def terrain_torch(torch, rows, col0, ncols, cols_total, seed, holes, device):
    g = torch.Generator(device="cpu")
    g.manual_seed(1234 + seed)
    ncomp = 14
    wl = 4.0 * (0.5 ** (torch.arange(ncomp, dtype=torch.float64) * (5.0 / (ncomp - 1))))  # 4 m .. 0.125 m
    ang = torch.rand(ncomp, generator=g, dtype=torch.float64) * (2 * np.pi)
    ph = torch.rand(ncomp, generator=g, dtype=torch.float64) * (2 * np.pi)
    amp = 0.05 * wl / wl[0] * 2.2
    length_x, length_y = rows * RES, cols_total * RES
    x = (0.5 * length_x - 0.5 * RES) - RES * torch.arange(rows, dtype=torch.float64)
    y = (0.5 * length_y - 0.5 * RES) - RES * torch.arange(col0, col0 + ncols, dtype=torch.float64)
    x = x.to(device)
    y = y.to(device)
    z = torch.zeros((ncols, rows), dtype=torch.float32, device=device)
    for k in range(ncomp):
        kx = float(2 * np.pi / wl[k] * torch.cos(ang[k]))
        ky = float(2 * np.pi / wl[k] * torch.sin(ang[k]))
        arg = (ky * y)[:, None] + (kx * x + float(ph[k]))[None, :]
        z += float(amp[k]) * torch.sin(arg).to(torch.float32)
    ii = torch.arange(rows, device=device, dtype=torch.int64)[None, :]
    jj = torch.arange(col0, col0 + ncols, device=device, dtype=torch.int64)[:, None]

    def h32(a, b, salt):
        h = (a * 73856093) ^ (b * 19349663) ^ (salt * 83492791 + seed * 2654435761)
        h = (h ^ (h >> 13)) * 1274126177
        h = h ^ (h >> 16)
        return h & 0x7FFFFFFF

    z += 1e-3 * ((h32(ii, jj, 1) % 20001).to(torch.float32) / 10000.0 - 1.0)  # +-1 mm sensor-like noise
    # raised rectangles (cliffs) and exactly flat patches on a 512-cell lattice
    ci, cj = ii // 512, jj // 512
    for salt, kind in ((2, "cliff"), (3, "flat")):
        oi = 32 + h32(ci, cj, salt) % 256
        oj = 32 + h32(ci, cj, salt + 10) % 256
        hi = 24 + h32(ci, cj, salt + 20) % 160
        hj = 24 + h32(ci, cj, salt + 30) % 160
        li, lj = ii - ci * 512, jj - cj * 512
        inside = (li >= oi) & (li < oi + hi) & (lj >= oj) & (lj < oj + hj) & (h32(ci, cj, salt + 40) % 4 < 2)
        if kind == "cliff":
            z = torch.where(inside, z + 0.2, z)
        else:
            z = torch.where(inside, torch.full_like(z, 0.125), z)
    if holes > 0:
        # one candidate blob (radius 4 cells, ~50 cells) per 64 x 64 block, kept with probability p
        p = min(1.0, holes * 4096.0 / 50.0)
        bi, bj = ii // 64, jj // 64
        oi = 8 + h32(bi, bj, 5) % 48
        oj = 8 + h32(bi, bj, 6) % 48
        keep = (h32(bi, bj, 7) % 10000) < int(p * 10000)
        li, lj = ii - bi * 64, jj - bj * 64
        hole = keep & (((li - oi) ** 2 + (lj - oj) ** 2) <= 16)
        z = torch.where(hole, torch.full_like(z, float("nan")), z)
    return z.contiguous()


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def wait_first(self, timeout=3.0):
        """nvidia-smi needs a few hundred ms to deliver its first line: the timed region starts after it."""
        t0 = time.perf_counter()
        while self.proc and not self.lines and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_name(rows, cols, holes):
    """The same string in both arms (`--impl b200` and `--impl reference`): the driver compares them."""
    return f"{rows}x{cols} elevation @ {RES} m, full filter chain (YAML parameters), {100 * holes:g} % NaN holes"


def host_cpu():
    """Model name and logical CPU count of the box (the CPU arms are only comparable on the same box)."""
    model = None
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    model = ln.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    return {"model": model, "logical_cpus": os.cpu_count(), "usable_threads": len(os.sched_getaffinity(0))}


def bench_map_crop(n, holes):
    """The top-left n x n crop of the 8192 x 8192 bench map (same generator and seed as the GPU arm, evaluated on the CPU)."""
    import torch
    z = terrain_torch(torch, 8192, 0, n, 8192, 3, holes, torch.device("cpu"))   # (n columns, 8192 rows)
    return np.asfortranarray(z[:, :n].numpy().T)


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def profile_traffic():
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "roofline_latest.json")) as f:
            return json.load(f)
    except Exception:
        return None


def run_reference(args):
    """`--impl reference`: the reference's own CPU algorithm for this path — its restatement in oracle/ (the ROS/Eigen
    sources cannot be built in this image) — on all host threads; every step is a bounded 2048 x 2048 sample of the map."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import binding as ob
    n = 2048 if args.rows == 0 else args.rows
    z = bench_map_crop(n, args.holes)
    g = ob.Geometry.make(n, n, RES)
    p = ob.ChainParams.yaml_defaults(0)
    threads = len(os.sched_getaffinity(0))  # all host threads, also under torchrun (which exports OMP_NUM_THREADS=1)
    # each step is one pass over the bounded sample; at most two warm-up passes, each takes seconds
    warmup = min(args.warmup, 2)
    for _ in range(warmup):
        ob.chain(g, p, z, nthreads=threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o = ob.chain(g, p, z, nthreads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"reference_" + name: layer for name, layer in o.items()})
    val = n * n * args.steps / dt / 1e6
    args.warmup = warmup
    out = {"impl": "reference", "metric": "Mcells/s full filter chain, synthetic elevation", "value": val, "unit": "Mcells/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
           "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64 compute / f32 layers",
           "data": "synthetic",
           "config": {"workload": workload_name(8192, 8192, args.holes),
                      "sample": f"top-left {n}x{n} crop of the same map (same generator and seed as the GPU arm) per step",
                      "holes": args.holes, "host": host_cpu()},
           "cpu_baseline": {"value": val, "unit": "Mcells/s", "cores": threads, "kind": "port",
                            "sample": f"{n}x{n} cells per step, {args.steps} steps, OpenMP over {threads} host threads; "
                                      "restated CPU chain (not the ROS/Eigen binary)"},
           "e2e": {"value": val, "unit": "Mcells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def run_plugin_chain(args, torch, dev):
    """`--workload plugin_chain`: end to end through the reference-facing boundary itself — the C++ plugin shells
    filters::{Slope,Step,Roughness}Filter<grid_map::GridMap>::update() driven like filters::FilterChain drives them under the
    UNCHANGED YAML (robot_filter_parameter.yaml:10-28), host GridMaps in and out, `mapOut = mapIn` copies included.  Timed twice:
    with the cross-plugin fusion registry (one te_chain launch per map) and with TE_B200_FUSE_CHAIN=0 (three stand-alone literal
    kernels, the round-1 behaviour)."""
    import tempfile
    plugin = os.path.join(ROOT, "traversability_estimation_b200", "plugin")
    subprocess.check_call(["make", "-C", plugin, "-s"])
    rows = cols = args.rows or 4096
    z = terrain_torch(torch, rows, 0, cols, cols, 3, args.holes, dev)
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "elev.bin")
        z.cpu().numpy().tofile(src)
        passes = args.steps
        for name, fuse in (("fused_registry", "1"), ("standalone_literal", "0")):
            env = dict(os.environ, TE_B200_FUSE_CHAIN=fuse)
            r = subprocess.run([os.path.join(plugin, "test_plugins"), "bench", str(rows), str(cols), repr(RES), src, str(passes)],
                               capture_output=True, text=True, env=env, timeout=1800)
            if r.returncode != 0:
                raise SystemExit("test_plugins bench failed: " + r.stdout[-500:] + r.stderr[-500:])
            line = [ln for ln in r.stdout.splitlines() if ln.startswith("PLUGIN_CHAIN")][-1]
            kv = dict(t.split("=") for t in line.split()[1:])
            res[name] = {"mean_ms": float(kv["mean_ms"]), "best_ms": float(kv["best_ms"]), "fused_launches": int(kv["launches"]),
                         "layers_from_cache": int(kv["served"]), "Mcells_per_s": rows * cols / (float(kv["mean_ms"]) * 1e-3) / 1e6}
    ms = res["fused_registry"]["mean_ms"]
    print(json.dumps({"metric": "Mcells/s full filter chain, synthetic elevation", "value": rows * cols / (ms * 1e-3) / 1e6,
                      "unit": "Mcells/s", "n_gpus": 1, "steps": passes, "warmup": 1, "ms_per_step": ms, "higher_is_better": True,
                      "scaling": "strong", "vs_baseline": None, "dtype": "f32 (f64 certified slow path)", "data": "synthetic",
                      "config": {"workload": f"{rows}x{cols} elevation through the C++ plugin shells (slopeFilter, stepFilter, roughnessFilter "
                                             "update() on host GridMaps, unchanged YAML)", "holes": args.holes},
                      "roofline": None, "cpu_baseline": None,
                      "e2e": {"value": rows * cols / (ms * 1e-3) / 1e6, "unit": "Mcells/s", "h2d_bytes_per_step": 4 * rows * cols,
                              "d2h_bytes_per_step": 16 * rows * cols, "note": "wall clock around the three update() calls"},
                      "plugin_chain": res, "gpu_launches": res["fused_registry"]["fused_launches"] * 3, "clocks": None}))


def run_other(args, torch, dist, te, world, rank, local, dev):
    """Secondary BASELINE configs: a batch of 256 independent 512 x 512 maps (sharded by map, no communication) and the
    circular footprint sweep over a 4096 x 4096 traversability layer."""
    ctx = te.Context(local)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)
    prm = te.ChainParams.yaml_defaults(0)
    if args.workload == "batched512":
        n_total, n = 256, 256 // world
        rows = cols = args.rows or 512
        g = te.Geometry.make(rows, cols, RES)
        z = torch.stack([terrain_torch(torch, rows, 0, cols, cols, 1000 + rank * n + k, args.holes, dev) for k in range(n)])
        outs = [torch.empty((n, cols, rows), dtype=torch.float32, device=dev) for _ in range(4)]
        cells = n_total * rows * cols
        name = f"{n_total} independent {rows}x{cols} maps, full fused chain, {n} maps per GPU"
        outputs = dict(zip(("slope", "step", "roughness", "traversability"), outs))

        def step():
            ctx.chain_batched(g, prm, n, z, *outs, te.MEM_DEVICE)
    elif args.workload == "slope8192":
        rows = cols = args.rows or 8192
        assert world == 1
        g = te.Geometry.make(rows, cols, RES)
        nz = torch.rand((cols, rows), dtype=torch.float32, device=dev) * 0.5 + 0.5
        out = torch.empty_like(nz)
        cells = rows * cols
        name = f"SlopeFilter only (te_slope) over a {rows}x{cols} surface_normal_z layer, 8 B/cell"
        outputs = {"slope": out}

        def step():
            ctx.slope(g, 1.0, nz, out, te.MEM_DEVICE)
    else:
        rows = cols = args.rows or 4096
        assert world == 1, "footprint bench is single-GPU"
        g = te.Geometry.make(rows, cols, RES)
        z = terrain_torch(torch, rows, 0, cols, cols, 5, args.holes, dev)
        lay = [torch.empty((cols, rows), dtype=torch.float32, device=dev) for _ in range(4)]
        ctx.chain(g, prm, z, *lay, te.MEM_DEVICE)
        fp = te.FootprintParams.yaml_defaults()
        if args.workload == "footprint4096_offset0":
            fp.offset = 0.0   # SURVEY.md §8(d) config 5, the other variant: no annulus between radiusMin and radiusMax
        out = torch.empty((cols, rows), dtype=torch.float32, device=dev)
        cells = rows * cols
        name = f"footprint sweep r=0.30 m offset={fp.offset:.2f} m over {rows}x{cols} traversability/slope/step/elevation"
        outputs = {"traversability_footprint": out}

        def step():
            ctx.footprint(g, fp, lay[3], lay[0], lay[1], z, out, te.MEM_DEVICE)
        if args.workload == "footprint_polygon4096":
            # traversabilityFootprint(yaw) with the YAML footprint (robot_footprint_parameter.yaml:3) and yaw (robot.yaml:9): two layers
            poly = [[0.45, 0.30], [0.45, -0.30], [-0.45, -0.30], [-0.45, 0.30]]
            out2 = torch.empty((cols, rows), dtype=torch.float32, device=dev)
            name = f"polygon footprint sweep (0.9 m x 0.6 m, yaw 0.7854: traversability_x + traversability_rot) over {rows}x{cols}"
            outputs = {"traversability_x": out, "traversability_rot": out2}

            def step():  # noqa: F811
                ctx.footprint_polygon(g, fp, poly, 0.7854, lay[3], lay[0], lay[1], z, out, out2, te.MEM_DEVICE)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    l0, _ = ctx.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs, dist, world, rank)
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    l1, _ = ctx.stats()
    if rank == 0:
        peak, src = measured_peak()
        bpc = 8 if args.workload == "slope8192" else (24 if args.workload == "footprint_polygon4096" else ALG_BYTES_PER_CELL)
        ach = bpc * (cells / world) / (ms / args.steps * 1e-3) / 1e9
        print(json.dumps({"metric": "Mcells/s " + {"batched512": "full filter chain", "slope8192": "slope filter"}.get(args.workload, "footprint sweep") + ", synthetic elevation",
                          "value": cells * args.steps / (ms * 1e-3) / 1e6, "unit": "Mcells/s", "n_gpus": world, "steps": args.steps,
                          "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong",
                          "vs_baseline": None, "dtype": "f32 (f64 certified slow path)" if args.workload == "batched512" else "f64/f32", "data": "synthetic",
                          "config": {"workload": name, "holes": args.holes},
                          "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
                                       "peak_source": src, "note": "whole step (all kernels of the pass), %d B/cell" % bpc},
                          "cpu_baseline": None, "e2e": None, "gpu_launches": int(l1 - l0), "clocks": None}))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    import traversability_estimation_b200 as te

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, (world, args.gpus)

    if args.workload == "plugin_chain":
        assert world == 1
        return run_plugin_chain(args, torch, dev)
    if args.workload in ("batched512", "footprint4096", "footprint4096_offset0", "footprint_polygon4096", "slope8192"):
        return run_other(args, torch, dist, te, world, rank, local, dev)
    rows = args.rows or {"chain8192": 8192, "chain2048": 2048}.get(args.workload, 8192)
    base_cols = args.cols or rows
    if args.scaling == "weak":
        cols_total, my_cols, col0 = base_cols * world, base_cols, base_cols * rank
    else:
        assert base_cols % world == 0
        cols_total, my_cols, col0 = base_cols, base_cols // world, (base_cols // world) * rank
    H = 4  # dependency radius of the YAML chain at 0.02 m (cells)
    hl = H if rank > 0 else 0
    hr = H if rank < world - 1 else 0

    g = te.Geometry.make(rows, cols_total, RES)
    prm = te.ChainParams.yaml_defaults(0)
    slab = te.Slab(col0, my_cols, hl, hr)
    ctx = te.Context(local)
    ctx.set_kernel({"auto": te.KERNEL_AUTO, "generic": te.KERNEL_GENERIC, "fused": te.KERNEL_FUSED}[args.kernel])
    stream = torch.cuda.Stream()  # a real stream: handle 0 (legacy default) would mean "the context's own stream"
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    own = terrain_torch(torch, rows, col0, my_cols, cols_total, 3, args.holes, dev)  # (my_cols, rows): column-major layer
    elev = torch.full((hl + my_cols + hr, rows), float("nan"), dtype=torch.float32, device=dev)
    elev[hl:hl + my_cols].copy_(own)
    # a pass touches 20 B/cell; when that fits the 126 MB L2, rotate through enough buffer sets that every timed pass
    # streams from HBM ("inputs larger than L2" by rotation instead of an explicit flush)
    pass_bytes = 20 * rows * my_cols
    nsets = 1 if pass_bytes > 3e8 else int(np.ceil(6e8 / pass_bytes))
    overlap = world > 1 and args.halo == "ipc" and args.halo_overlap != 0
    if overlap:
        nsets = max(nsets, 2)   # the halo columns of one set are rewritten while the chain reads another
    elevs = [elev] + [elev.clone() for _ in range(nsets - 1)]
    outsets = [[torch.empty((my_cols, rows), dtype=torch.float32, device=dev) for _ in range(4)] for _ in range(nsets)]
    outs = outsets[0]
    rot = [0]

    from traversability_estimation_b200.sharding import PeerHalo, SlabPlan, exchange_halo
    plan = SlabPlan(rank, world, cols_total, col0, my_cols, hl, hr)
    # halo exchange inside the step: peer-mapped pull through the C ABI (default) or NCCL send/recv.  With rotated buffer sets
    # (small slabs) each set has its own mapping.
    peers = [PeerHalo(dist, ctx, te, e, plan) for e in elevs] if (world > 1 and args.halo == "ipc") else None
    if peers:
        torch.cuda.synchronize()
        for ph in peers:
            ph.publish()      # the owned columns are in place (the bench map is static)
        ctx.synchronize()
        dist.barrier()        # host-side ordering: every rank's ready event is recorded before anyone waits on it
    hev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)] if world > 1 else []
    timed = [False, 0]
    # overlapped exchange: a step still pulls one halo and runs one chain, but the pull it issues is the NEXT buffer set's, on a
    # side stream, ordered by events (pulled[k]: the halo of set k is in place; done[k]: the last chain on set k has read it)
    side = torch.cuda.Stream() if overlap else None
    pulled = [torch.cuda.Event() for _ in range(nsets)] if overlap else []
    done = [torch.cuda.Event() for _ in range(nsets)] if overlap else []

    def pull_async(k):
        side.wait_event(done[k])
        ctx.set_stream(side.cuda_stream)
        rec = timed[0] and timed[1] < len(hev)
        if rec:
            hev[timed[1]][0].record(side)
        peers[k].pull(g)
        if rec:
            hev[timed[1]][1].record(side)
            timed[1] += 1
        pulled[k].record(side)
        ctx.set_stream(stream.cuda_stream)

    if overlap:
        for e in done:
            e.record(stream)
        pull_async(0)

    def exchange():
        if world == 1:
            return
        k = rot[0] % nsets
        rec = timed[0] and timed[1] < len(hev)
        if rec:
            hev[timed[1]][0].record(stream)
        if peers:
            peers[k].pull(g)
        else:
            exchange_halo(dist, elevs[k], plan, H)
        if rec:
            hev[timed[1]][1].record(stream)
            timed[1] += 1

    def step():
        k = rot[0] % nsets
        if overlap:
            stream.wait_event(pulled[k])
        else:
            exchange()
        rot[0] += 1
        o = outsets[k]
        ctx.chain(g, prm, elevs[k], o[0], o[1], o[2], o[3], te.MEM_DEVICE, slab=slab)
        if overlap:
            done[k].record(stream)
            pull_async((k + 1) % nsets)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    if rank == 0:
        sampler.wait_first()  # the timed region starts only once nvidia-smi delivers samples
    launches0, _ = ctx.stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    timed[0] = True
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    timed[0] = False
    ms_total = ev0.elapsed_time(ev1)
    halo_ms = (sum(a.elapsed_time(b) for a, b in hev[:timed[1]]) / max(timed[1], 1)) if world > 1 else 0.0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        last = outsets[(rot[0] - 1) % nsets]
        dump_outputs(args.dump_outputs, dict(zip(("slope", "step", "roughness", "traversability"), last)), dist, world, rank)
    launches1, slow_cells = ctx.stats()
    # kernel split (fused stencil / fix-up tiers): CUDA events recorded inside the C ABI around the launches, in a SEPARATE short
    # run of the same step — events between the kernels would serialise the programmatic dependent launches of the timed region
    ctx.timing()  # drop anything accumulated
    ctx.enable_timing(True)
    for _ in range(min(args.steps, 20)):
        step()
    barrier()
    main_ms, fix_ms, nlaunch = ctx.timing()
    ctx.enable_timing(False)
    t = torch.tensor([ms_total, main_ms / max(nlaunch, 1), fix_ms / max(nlaunch, 1), halo_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, main_avg, fix_avg, halo_ms = (float(v) for v in t.tolist())
    cells_total = rows * cols_total
    value = cells_total * args.steps / (ms_total * 1e-3) / 1e6

    # ---- end-to-end through the C ABI with HOST (pinned) buffers: H2D + kernels + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        h_in = torch.empty((hl + my_cols + hr, rows), dtype=torch.float32).pin_memory()
        h_in.copy_(elev)
        h_out = [torch.empty((my_cols, rows), dtype=torch.float32).pin_memory() for _ in range(4)]
        ctx.set_stream(None)
        nsteps_e2e = max(3, min(args.steps, 10))
        for _ in range(2):
            ctx.chain(g, prm, h_in.data_ptr(), *[o.data_ptr() for o in h_out], te.MEM_HOST, slab=slab)
        barrier()
        t0 = time.perf_counter()
        for _ in range(nsteps_e2e):
            ctx.chain(g, prm, h_in.data_ptr(), *[o.data_ptr() for o in h_out], te.MEM_HOST, slab=slab)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": cells_total * nsteps_e2e / float(dt) / 1e6, "unit": "Mcells/s",
               "h2d_bytes_per_step": int(h_in.numel() * 4 * world), "d2h_bytes_per_step": int(4 * my_cols * rows * 4 * world),
               "steps": nsteps_e2e, "note": "te_chain(TE_MEM_HOST) from pinned host layers; slab + halo taken from the host map"}
        ctx.set_stream(stream.cuda_stream)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- CPU baseline: the oracle (restated reference chain) on a bounded crop of the same map, host threads
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import binding as ob
        n = min(2048, rows, my_cols)
        crop = np.asfortranarray(own[:n, :n].cpu().numpy().T)
        og = ob.Geometry.make(n, n, RES)
        op = ob.ChainParams.yaml_defaults(0)
        threads = len(os.sched_getaffinity(0))
        ob.chain(ob.Geometry.make(128, 128, RES), op, np.asfortranarray(crop[:128, :128]), nthreads=threads)  # warm the thread pool
        t0 = time.perf_counter()
        ob.chain(og, op, crop, nthreads=threads)
        dt = time.perf_counter() - t0
        n1 = min(512, n)   # SURVEY.md §8(d)-i: the reference is single-threaded per filter; one thread on a smaller crop
        c1 = np.asfortranarray(crop[:n1, :n1])
        t0 = time.perf_counter()
        ob.chain(ob.Geometry.make(n1, n1, RES), op, c1, nthreads=1)
        dt1 = time.perf_counter() - t0
        cpu = {"value": n * n / dt / 1e6, "unit": "Mcells/s", "cores": threads, "kind": "port",
               "sample": f"{n}x{n} crop of the same map, one pass, OpenMP over {threads} host threads "
                         f"({dt:.2f} s); restated CPU chain, not the ROS/Eigen binary",
               "single_thread": {"value": n1 * n1 / dt1 / 1e6, "unit": "Mcells/s", "cores": 1,
                                 "sample": f"{n1}x{n1} crop of the same map, one pass, one thread ({dt1:.2f} s)"},
               "host": host_cpu()}

    peak, peak_src = measured_peak()
    cells_per_launch = rows * my_cols
    achieved = ALG_BYTES_PER_CELL * cells_per_launch / (main_avg * 1e-3) / 1e9 if main_avg > 0 else None
    prof = profile_traffic()
    # the committed ncu capture is of one launch over an 8192 x 8192 slab with the fused kernel: quote it only there
    traffic = (prof or {}).get("dram_bytes_per_launch") if (rows == 8192 and my_cols == 8192 and args.kernel != "generic") else None
    out = {
        "metric": "Mcells/s full filter chain, synthetic elevation", "value": value, "unit": "Mcells/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32 (f64 certified slow path)",
        "data": "synthetic",
        "config": {"workload": workload_name(rows, cols_total, args.holes),
                   "tiling": f"{world} column slab(s) of {rows}x{my_cols}" +
                             ((" + 4-column halo, " + (("peer-mapped pull over NVLink (te_halo_pull, CUDA IPC)" + (", the next buffer set's pull overlapped on a side stream" if overlap else "")) if args.halo == "ipc" else "NCCL send/recv"))
                              if world > 1 else ""),
                   "holes": args.holes, "kernel": args.kernel,
                   "l2": ("working set %.2f GB/GPU per pass > 126 MB L2, no flush needed" % (pass_bytes / 1e9)) if nsets == 1 else
                         ("%d buffer sets rotated (%.0f MB total) so every pass streams from HBM" % (nsets, nsets * pass_bytes / 1e6)),
                   "slow_path_cells_per_launch": int(slow_cells)},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None,
                     "traffic": traffic, "peak_source": peak_src,
                     "kernel": "k_chain_fused" if args.kernel != "generic" else "k_chain_generic",
                     "kernel_ms": main_avg, "fixup_kernel_ms": fix_avg,
                     "algorithmic_bytes_per_launch": ALG_BYTES_PER_CELL * cells_per_launch,
                     # the four layers are final only after the fix-up tiers: the whole device step against the same peak
                     "step": {"ms": ms_total / args.steps, "achieved": ALG_BYTES_PER_CELL * cells_per_launch / (ms_total / args.steps * 1e-3) / 1e9,
                              "frac": ALG_BYTES_PER_CELL * cells_per_launch / (ms_total / args.steps * 1e-3) / 1e9 / peak}},
        "halo_ms": halo_ms if world > 1 else None,
        "halo": (args.halo if world > 1 else None),
        "cpu_baseline": cpu,
        "e2e": e2e,
        "gpu_launches": int(launches1 - launches0),
        "clocks": clocks,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
