"""Cost of the posterior variability maps accumulated inside the fused chain runner (icp_chain_set_statistics) on the bench
workload (femur GPMM-100 twin, config-1 mixture, bench.py's chains and initial states):

  off       device ms per step with statistics off. With --baseline-tag TAG the same measurement alternates, in separate
            processes, between this library and icp-proposal_b200/libicpcuda_TAG.so (a build of another revision copied
            there), so that the off path can be compared with the revision before the feature.
  on        device ms per step with statistics on at take_every_n 1, 10 and 50 (burn-in 0, normals on).
  e2e       a run of --e2e-steps steps, then the maps of every 50th record pooled over all chains: log_theta to the host plus
            icp_posterior_variability over the selected rows, against the maps read from the run (icp_chain_statistics).

Prints one JSON object per arm and a summary; writes them to --out when given. The card's name and power limit are
recorded with the numbers."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def setup(C):
    import ctypes

    import bench
    from icp_proposal_b200 import _lib, core
    if os.environ.get("ICPCUDA_LIB_TAG"):   # a build of an older revision: bind only the entry points it has
        have = ctypes.CDLL(_lib.LIB_PATH)
        for name in [n for n in _lib._SIGS if not hasattr(have, n)]:
            del _lib._SIGS[name]
    m, tv, tc, ids, eids, tp = bench.workload()
    ctx = core.Context(0)
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, tv, tc)
    ru = _lib.RANK_UPDATE_INT8
    pt = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, rank_update=ru)
    pm = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=ru)
    comps = [dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pt), dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pm),
             dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
    chain = core.Chain(model, tgt, comps, ev, max_chains=C)
    return dict(model=model, chain=chain, th0=bench.init_thetas(m, C), keep=(ctx, tgt, pt, pm, ev))


def timed(s, steps, warmup, stats=None):
    """ms per step of `steps` resumed steps after a run of `warmup` steps from theta0 (statistics set before it)."""
    import torch
    chain, C = s["chain"], len(s["th0"])
    if stats is not None:
        chain.set_statistics(*stats)
    th0 = torch.from_numpy(s["th0"]).cuda()
    chain.run_device(C, warmup, th0.data_ptr(), seed=1024)
    chain.run_device(C, steps, None, seed=1024)
    ms, launches = chain.last_run_stats()
    return ms / steps, launches / steps


def arm_off(args):
    s = setup(args.chains)
    ms, per_step = timed(s, args.steps, args.warmup)
    lib = os.environ.get("ICPCUDA_LIB_TAG") or "product"
    return dict(arm="off", lib=lib, chains=args.chains, steps=args.steps, ms_per_step=ms, kernels_per_step=per_step)


def arm_on(args):
    s = setup(args.chains)
    out = dict(arm="on", chains=args.chains, steps=args.steps)
    out["off_ms_per_step"], _ = timed(s, args.steps, args.warmup, None)
    for n in (1, 10, 50):
        ms, per_step = timed(s, args.steps, args.warmup, (0, n, 0, True))
        out[f"every_{n}_ms_per_step"] = ms
        out[f"every_{n}_overhead"] = ms / out["off_ms_per_step"] - 1.0
        out[f"every_{n}_kernels_per_step"] = per_step
        s["chain"].set_statistics(None)
    return out


def arm_e2e(args):
    from icp_proposal_b200 import core
    s = setup(args.chains)
    chain, model, th0 = s["chain"], s["model"], s["th0"]
    C, n, every = len(th0), args.e2e_steps, 50
    L = model.K + 10
    chain.run(th0[:, :], 2, seed=3, log_theta=False)     # sizes the workspaces, captures the step graph
    # (a) chain log on the host, then icp_posterior_variability over the selected rows
    t0 = time.perf_counter()
    run = chain.run(th0, n, seed=1024, log_theta=True)
    t1 = time.perf_counter()
    sel = run["theta"][::every].reshape(-1, L)
    want = core.posterior_variability(model, sel, True)
    t2 = time.perf_counter()
    del run
    # (b) the maps accumulated inside the run
    chain.set_statistics(0, every, 0, True)
    chain.run(th0, 2, seed=3, log_theta=False)
    t3 = time.perf_counter()
    chain.run(th0, n, seed=1024, log_theta=False)
    t4 = time.perf_counter()
    got = chain.statistics(-1, True)
    t5 = time.perf_counter()
    dev = {k: float(np.max(np.abs(got[k] - want[k])) / np.max(np.abs(want[k]))) for k in ("mean", "cov", "total_variance", "normal_variance")}
    return dict(arm="e2e", chains=C, steps=n, take_every_n=every, samples=int(got["n"]), log_samples=len(sel),
                log_run_s=t1 - t0, log_variability_s=t2 - t1, log_total_s=t2 - t0, log_theta_bytes=n * C * L * 8,
                stream_run_s=t4 - t3, stream_read_s=t5 - t4, stream_total_s=t5 - t3,
                max_deviation_relative_to_map_max=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chains", type=int, default=4736)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=1000)
    ap.add_argument("--baseline-tag", default=None, help="alternate the off arm with libicpcuda_TAG.so")
    ap.add_argument("--repeats", type=int, default=2, help="alternations of the off arm")
    ap.add_argument("--arms", default="off,on,e2e")
    ap.add_argument("--arm", default=None, help=argparse.SUPPRESS)   # one arm in this process
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if args.arm:
        print(json.dumps({"off": arm_off, "on": arm_on, "e2e": arm_e2e}[args.arm](args)), flush=True)
        return
    results = dict(card=card())
    print(json.dumps(results), flush=True)

    def child(arm, tag=None):
        env = dict(os.environ)
        env.pop("ICPCUDA_LIB_TAG", None)
        if tag:
            env["ICPCUDA_LIB_TAG"] = tag
        cmd = [sys.executable, os.path.abspath(__file__), "--arm", arm, "--chains", str(args.chains), "--steps", str(args.steps),
               "--warmup", str(args.warmup), "--e2e-steps", str(args.e2e_steps)]
        r = subprocess.run(cmd, env=env, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"{arm} ({tag or 'product'}) failed:\n{r.stdout}\n{r.stderr}")
        res = json.loads(r.stdout.strip().splitlines()[-1])
        print(json.dumps(res), flush=True)
        return res

    arms = args.arms.split(",")
    if "off" in arms:
        runs = []
        for _ in range(args.repeats):
            runs.append(child("off"))
            if args.baseline_tag:
                runs.append(child("off", args.baseline_tag))
        results["off"] = runs
        by = {}
        for r in runs:
            by.setdefault(r["lib"], []).append(r["ms_per_step"])
        results["off_ms_per_step"] = {k: dict(min=min(v), max=max(v), runs=v) for k, v in by.items()}
    if "on" in arms:
        results["on"] = child("on")
    if "e2e" in arms:
        results["e2e"] = child("e2e")
    print(json.dumps(results), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
