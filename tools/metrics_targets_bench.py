"""The scoring stage of config 4 (StdIcpVsChainICPrandomInitComparisonAll.scala:43-47) over a target set; prints one JSON object.

For G = 1, 8, 24 and 47 targets (the perturbed femur-twin targets of tests/test_gpu_multi_target.py, GPMM-100) x 300 rows
(the random inits of bench.init_thetas, each shifted by a random translation so that the measures are not trivial), the
registration measures and the Dice coefficient (10 000 seeded samples) are taken two ways:
    loop     G single-target calls back to back, one per target on that target's rows (the only way before target sets)
    targets  one icp_registration_metrics_targets / icp_dice_coefficient_targets call over all rows
wall ms: median host time of a pass (every call synchronises); device ms: the sum of the CUDA kernel and copy durations of
one pass, from torch.profiler in a pass of its own. Every row of the two ways is checked bit for bit. The GPU name, power
limit and maximum SM clock are read in the same run.

Usage: python tools/metrics_targets_bench.py [--out FILE] [--repeats R] [--groups 1,8,24,47] [--rows 300]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from icp_proposal_b200 import core, synth  # noqa: E402

N_SAMPLES = 10000


def _gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _device_ms(fn):
    """Sum of the CUDA activity durations (kernels, copies) of one call of fn."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as p:
        fn()
    return sum(e.time_range.elapsed_us() for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA) * 1e-3


def _timed(fn, repeats):
    out = fn()                                                   # warm-up
    wall = []
    for _ in range(repeats):
        t = time.perf_counter()
        fn()
        wall.append((time.perf_counter() - t) * 1e3)
    return out, float(np.median(wall)), _device_ms(fn)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--groups", default="1,8,24,47")
    ap.add_argument("--rows", type=int, default=300)
    args = ap.parse_args()
    groups = [int(g) for g in args.groups.split(",")]
    g = os.path.join(ROOT, "tests", "golden")
    meshes, gp = np.load(os.path.join(g, "femur_meshes.npz")), np.load(os.path.join(g, "femur_gpmm_100.npz"))
    base = dict(ref=meshes["ref"].astype(np.float64), cells=meshes["cells"].astype(np.int32),
                basis=gp["basis"].astype(np.float64), variance=gp["variance"].astype(np.float64))
    K = len(base["variance"])
    ctx = core.Context(0)
    model = core.Model(ctx, base["ref"], base["cells"], base["basis"], base["variance"])
    tgts = []
    for t in range(max(groups)):
        tv = synth.model_instance(base, np.random.default_rng(100 + t).normal(0, 1.0, K))
        tgts.append(core.Target(ctx, tv + np.random.default_rng(7 + t).normal(0, 0.5, tv.shape), base["cells"]))
    result = dict(gpu=_gpu_info(), rows_per_target=args.rows, dice_samples=N_SAMPLES, repeats=args.repeats, groups=[])
    for G in groups:
        C = G * args.rows
        th = bench.init_thetas(base, C)
        th[:, 1:4] += np.random.default_rng(5).normal(0, 2.0, (C, 3))
        tidx = np.repeat(np.arange(G), args.rows)
        sets = tgts[:G]
        rows = [np.flatnonzero(tidx == t) for t in range(G)]

        def loop_metrics():
            out = np.empty((C, 4))
            for t in range(G):
                out[rows[t]] = core.registration_metrics(model, sets[t], th[rows[t]])
            return out

        def loop_dice():
            out = np.empty(C)
            for t in range(G):
                out[rows[t]] = core.dice_coefficient(model, sets[t], th[rows[t]], n_samples=N_SAMPLES)
            return out

        row = dict(targets=G, rows=C)
        for name, loop, batched in (
                ("metrics", loop_metrics, lambda: core.registration_metrics(model, sets, th, target_index=tidx)),
                ("dice", loop_dice, lambda: core.dice_coefficient(model, sets, th, n_samples=N_SAMPLES, target_index=tidx))):
            a, wa, da = _timed(loop, args.repeats)
            b, wb, db = _timed(batched, args.repeats)
            same = bool(np.array_equal(a, b, equal_nan=True))
            assert same, f"G = {G} {name}: the target-set call differs from the per-target calls"
            row[name] = dict(loop=dict(wall_ms=wa, device_ms=da), targets=dict(wall_ms=wb, device_ms=db),
                             wall_speedup=wa / wb, device_speedup=da / db, bit_identical=same)
        result["groups"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
    for t in tgts:
        t.close()
    model.close()
    ctx.close()
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
