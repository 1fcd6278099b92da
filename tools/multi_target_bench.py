"""Chains against many targets in one device-resident run (icp_chain_create_targets) on the shape of BASELINE config 4
(StdIcpVsChainICPrandomInitComparisonAll: targets x 100 random inits, Hausdorff evaluator Exponential(100), the config-1
mixture, INT8 rank update), for G = 1, 8, 24 and 47 perturbed femur-twin targets, measured three ways:
  multi      one multi-target run of G x 100 chains
  loop       G single-target runs of 100 chains back to back (one handle per target, the workaround without target sets)
  single     one single-target run of G x 100 chains (the rate at equal chain count, one target)
samples/s = chains x steps / device time of the run(s) (icp_chain_last_run_stats); the loop also reports host wall time, which
adds its per-run synchronisations. Every handle is warmed up (graph capture, look-ahead probing) before the timed run.
    python tools/multi_target_bench.py [--steps 20] [--groups 1,8,24,47] [--out profiles/multi_target_bench.json]
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
from icp_proposal_b200 import _lib, core, synth  # noqa: E402

INITS = 100


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        return name, float(q[0]), float(q[1])
    except Exception:   # noqa: BLE001 - no nvidia-smi: the card's name is still recorded
        return name, None, None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--groups", default="1,8,24,47")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    groups = [int(g) for g in args.groups.split(",")]
    m, _, _, ids, _, _ = bench.workload()
    K = bench.K_RANK
    ctx = core.Context(0)
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    handles, entries = [], []
    for g in range(max(groups)):
        # the perturbed targets of test_config4_hausdorff_chains_on_perturbed_targets
        tv = synth.model_instance(m, np.random.default_rng(100 + g).normal(0, 1.0, K))
        tv = tv + np.random.default_rng(7 + g).normal(0, 0.5, tv.shape)
        tgt = core.Target(ctx, tv, m["cells"])
        tp = tv[:: len(tv) // (2 * K)][: 2 * K]
        mk = lambda d: core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, d, True, ids, tp, rank_update=_lib.RANK_UPDATE_INT8)
        pt, pm = mk(_lib.TARGET_SAMPLING), mk(_lib.MODEL_SAMPLING)
        comps = [dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pt), dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pm),
                 dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
        ev = core.Evaluator(model, tgt, _lib.EVAL_HAUSDORFF, 0, True, 100.0)
        entries.append((tgt, comps, ev, len(tv)))
        handles += [ev, pt, pm, tgt]
    steps = args.steps
    name, power, clock = gpu_info()
    out = {"gpu": name, "power_limit_w": power, "max_sm_clock_mhz": clock, "steps": steps, "inits_per_target": INITS,
           "workload": "config 4 shape: femur twin N=1622 K=101, perturbed targets, config-1 mixture, Hausdorff, INT8", "groups": {}}

    def timed(chain, th0, tidx=None):
        chain.run(th0, steps, seed=5, log_theta=False, target_index=tidx)        # warm-up: graphs, look-ahead widths
        t0 = time.perf_counter()
        r = chain.run(th0, steps, seed=6, log_theta=False, target_index=tidx)
        wall = time.perf_counter() - t0
        return chain.last_run_stats()[0], wall, float(r["n_accepted"].mean() / steps)

    for G in groups:
        C = G * INITS
        th0 = np.concatenate([bench.init_thetas(m, INITS) for _ in range(G)])
        tidx = np.repeat(np.arange(G), INITS)
        res = {"chains": C}
        # (1) one multi-target run
        ents = [e[:3] for e in entries[:G]]
        ch = core.Chain(model, targets=ents, max_chains=C) if G > 1 else core.Chain(model, *ents[0], C)
        ms, wall, acc = timed(ch, th0, tidx if G > 1 else None)
        ch.close()
        res["multi"] = {"samples_per_s": C * steps / (ms * 1e-3), "device_ms": ms, "wall_s": wall, "accept_rate": acc}
        # (2) G single-target runs of 100 chains back to back
        chains = [core.Chain(model, *entries[g][:3], INITS) for g in range(G)]
        for c in chains:
            c.run(th0[:INITS], steps, seed=5, log_theta=False)
        ms_sum, t0 = 0.0, time.perf_counter()
        for c in chains:
            c.run(th0[:INITS], steps, seed=6, log_theta=False)
            ms_sum += c.last_run_stats()[0]
        wall = time.perf_counter() - t0
        for c in chains:
            c.close()
        res["loop"] = {"samples_per_s": C * steps / (ms_sum * 1e-3), "device_ms": ms_sum, "wall_s": wall,
                       "samples_per_s_wall": C * steps / wall}
        # (3) one single-target run of G x 100 chains
        ch = core.Chain(model, *entries[0][:3], C)
        ms, wall, acc = timed(ch, th0)
        ch.close()
        res["single"] = {"samples_per_s": C * steps / (ms * 1e-3), "device_ms": ms, "wall_s": wall, "accept_rate": acc}
        # Hausdorff target -> model lists are padded to the largest vertex count of the set: wasted queries / all queries
        nts = np.array([entries[g][3] for g in range(G)])
        res["padded_query_fraction"] = float((nts.max() - nts).sum() / (nts.max() * G))
        res["multi_over_loop"] = res["multi"]["samples_per_s"] / res["loop"]["samples_per_s"]
        res["multi_over_single"] = res["multi"]["samples_per_s"] / res["single"]["samples_per_s"]
        out["groups"][str(G)] = res
        print(json.dumps({"G": G, **res}), flush=True)
    for h in handles:
        h.close()
    model.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
