"""Deterministic-ICP runner (icp_std_icp_*) on the workloads that use IcpBasedSurfaceFitting.runfitting; prints one JSON object.

- BASELINE config 2 (IcpRegistration.scala:40-43): femur GPMM-50, n = N = 1622 points per direction, sigma2 = 1e-15, step 1,
  101 iterations, one fit: all model sampling, all target sampling, alternating. Iterations/s and closest-point queries/s of
  the runner (device time, icp_std_icp_last_run_stats), launches per iteration, the wall-clock iterations/s of the per-call
  loop (icp_std_icp_iteration from Python, as api.IcpBasedSurfaceFitting ran it before) on the same inputs, and per row the
  largest |delta alpha| between the runner and the per-call iteration applied to the runner's previous row.
- The ICP arm of config 4 (StdIcpVsChainICPrandomInitComparisonAll.scala:148): 100 random inits x 101 iterations, Philox coin,
  GPMM-100 and GPMM-200.
- 2368 fits of GPMM-100 in one batch: fits/s.
- config4_icp_arm_targets: the ICP arm of config 4 over G = 1, 8, 24 and 47 targets (the perturbed femur-twin targets of
  tools/multi_target_bench.py, each with its own 1622 target points) x 100 fits, GPMM-100 and GPMM-200, measured three ways:
    multi   one run of a target-set handle (icp_std_icp_create_targets) with G x 100 fits
    loop    G single-target runs of 100 fits back to back (one handle per target: the only way before target sets)
    single  one single-target run of G x 100 fits (the rate at equal fit count on one target)
  fits/s from device time (the loop: the sum of its runs' device times; its wall time adds the per-run synchronisations),
  launches per iteration, and whether every multi fit equals its loop fit bit for bit.

Usage: python tools/std_icp_bench.py [--out FILE] [--repeats R] [--groups 1,8,24,47]
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
from icp_proposal_b200 import _lib, core, synth  # noqa: E402

N = 1622
ITERS = 101


def _gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def _load():
    g = os.path.join(ROOT, "tests", "golden")
    meshes = np.load(os.path.join(g, "femur_meshes.npz"))
    out = dict(ref=meshes["ref"].astype(np.float64), cells=meshes["cells"].astype(np.int32),
               target=meshes["target_aligned"].astype(np.float64), target_cells=meshes["target_cells"].astype(np.int32))
    for k in ("50", "100", "200"):
        z = np.load(os.path.join(g, f"femur_gpmm_{k}.npz"))
        out[k] = (z["basis"].astype(np.float64), z["variance"].astype(np.float64))
    return out


def _timed(runner, th0, sig, n_it, repeats, **kw):
    runner.run(th0, sig, n_it, **kw)                    # warm-up: captures the iteration graphs
    ms, wall = [], []
    out = None
    for _ in range(repeats):
        t = time.perf_counter()
        out = runner.run(th0, sig, n_it, **kw)
        wall.append(time.perf_counter() - t)
        d, launches = runner.last_run_stats()
        ms.append(d)
    return out, float(np.median(ms)), float(np.median(wall)), launches


INITS = 100


def targets_section(ctx, fx, models, ids, groups, repeats):
    """config4_icp_arm_targets (see the module docstring)."""
    base = dict(ref=fx["ref"], basis=fx["100"][0], variance=fx["100"][1])
    K100 = len(base["variance"])
    tgts, tps = [], []
    for g in range(max(groups)):
        # the perturbed targets of tools/multi_target_bench.py
        tv = synth.model_instance(base, np.random.default_rng(100 + g).normal(0, 1.0, K100))
        tv = tv + np.random.default_rng(7 + g).normal(0, 0.5, tv.shape)
        tgts.append(core.Target(ctx, tv, fx["cells"]))
        tps.append(synth.near_surface_queries(tv, fx["cells"], N, seed=1024, sd=0.0))
    out = []
    for k in ("100", "200"):
        m = models[k]
        for G in groups:
            C = G * INITS
            th = np.zeros((C, m.K + 10)); th[:, 0] = 1.0
            th[:, 10:] = np.random.default_rng(4).normal(0, 1.0, (C, m.K))     # random inits
            tidx = np.repeat(np.arange(G), INITS)
            row = dict(K=m.K, targets=G, fits=C, iterations=ITERS)
            multi = core.StdIcp(m, model_point_ids=ids, direction=_lib.MODEL_AND_TARGET_SAMPLING, max_fits=C,
                                targets=list(zip(tgts[:G], tps[:G]))) if G > 1 else \
                core.StdIcp(m, tgts[0], ids, tps[0], 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=C)
            kw = dict(seed=7, log=False, target_index=tidx) if G > 1 else dict(seed=7, log=False)
            mo, ms, wall, launches = _timed(multi, th, (1e-15,), ITERS - 1, repeats, **kw)
            multi.close()
            row["multi"] = dict(device_ms=ms, fits_per_s=C / (ms * 1e-3), launches_per_iteration=launches / ITERS, wall_ms=wall * 1e3)
            # the loop: one handle per target, each warmed up, then the G runs back to back
            hs = [core.StdIcp(m, tgts[g], ids, tps[g], 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=INITS) for g in range(G)]
            for g, h in enumerate(hs):
                h.run(th[g * INITS:(g + 1) * INITS], (1e-15,), ITERS - 1, seed=7, fit_id_offset=g * INITS, log=False)
            best = None
            for _ in range(repeats):
                t = time.perf_counter()
                lo, lms, ll = [], 0.0, 0
                for g, h in enumerate(hs):
                    lo.append(h.run(th[g * INITS:(g + 1) * INITS], (1e-15,), ITERS - 1, seed=7, fit_id_offset=g * INITS, log=False))
                    d, n = h.last_run_stats()
                    lms += d; ll += n
                lwall = time.perf_counter() - t
                if best is None or lms < best[0]:
                    best = (lms, lwall, ll)
            for h in hs:
                h.close()
            lms, lwall, ll = best
            row["loop"] = dict(device_ms=lms, fits_per_s=C / (lms * 1e-3), launches_per_iteration=ll / ITERS, wall_ms=lwall * 1e3,
                               wall_fits_per_s=C / lwall)
            row["multi_equals_loop"] = bool(np.array_equal(mo["alpha_final"], np.concatenate([o["alpha_final"] for o in lo])) and
                                            np.array_equal(mo["status"], np.concatenate([o["status"] for o in lo])))
            one = core.StdIcp(m, tgts[0], ids, tps[0], 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=C)
            _, sms, swall, sl = _timed(one, th, (1e-15,), ITERS - 1, repeats, seed=7, log=False)
            one.close()
            row["single"] = dict(device_ms=sms, fits_per_s=C / (sms * 1e-3), launches_per_iteration=sl / ITERS, wall_ms=swall * 1e3)
            row["multi_vs_loop_device"] = lms / ms
            row["multi_vs_loop_wall"] = lwall / wall
            row["multi_vs_single_device"] = sms / ms
            row["failed_fits"] = int((mo["status"] != 0).sum())
            print(json.dumps(row), file=sys.stderr, flush=True)
            out.append(row)
    for t in tgts:
        t.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--groups", default="1,8,24,47")
    a = ap.parse_args()
    fx = _load()
    ctx = core.Context(0)
    res = dict(device=_gpu_info(), version=ctx.version(), repeats=a.repeats)
    tgt = core.Target(ctx, fx["target"], fx["target_cells"])
    rng = np.random.default_rng(1024)
    ids = rng.integers(0, N, N)
    tp = synth.near_surface_queries(fx["target"], fx["target_cells"], N, seed=1024, sd=0.0)
    models = {k: core.Model(ctx, fx["ref"], fx["cells"], *fx[k]) for k in ("50", "100", "200")}

    # ---- config 2 ----
    model = models["50"]
    K = model.K
    th0 = model.theta(center=(0, 0, 0))[None]
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=1)
    cfg2 = {}
    for name, dirs in (("model_sampling", np.zeros(ITERS, np.int32)), ("target_sampling", np.ones(ITERS, np.int32)),
                       ("alternating", (np.arange(ITERS) % 2).astype(np.int32))):
        out, ms, wall, launches = _timed(runner, th0, (1e-15,), ITERS - 1, a.repeats, directions=dirs.reshape(-1, 1))
        # the per-call loop, wall clock, same inputs (one warm-up iteration of each direction first)
        for d in (0, 1):
            core.std_icp_iteration(model, tgt, d, ids, tp, 1e-15, 1.0, np.zeros((1, K)))
        t = time.perf_counter()
        alpha = np.zeros((1, K))
        for d in dirs:
            alpha = core.std_icp_iteration(model, tgt, int(d), ids, tp, 1e-15, 1.0, alpha)
        per_call_s = time.perf_counter() - t
        # row by row: the per-call iteration from the runner's previous row
        rows = out["log_alpha"][:, 0]
        delta = []
        for it, d in enumerate(dirs):
            prev = np.zeros((1, K)) if it == 0 else rows[it - 1][None]
            delta.append(float(np.abs(core.std_icp_iteration(model, tgt, int(d), ids, tp, 1e-15, 1.0, prev)[0] - rows[it]).max()))
        its = ITERS / (ms * 1e-3)
        cfg2[name] = dict(device_ms=ms, iterations_per_s=its, cp_queries_per_s=its * N, launches_per_iteration=launches / ITERS,
                          runner_wall_ms=wall * 1e3, runner_wall_iterations_per_s=ITERS / wall,
                          per_call_wall_ms=per_call_s * 1e3, per_call_wall_iterations_per_s=ITERS / per_call_s,
                          speedup_device_vs_per_call_wall=its / (ITERS / per_call_s),
                          speedup_wall_vs_per_call_wall=per_call_s / wall,
                          max_abs_dalpha=max(delta), max_abs_alpha=float(np.abs(rows).max()), max_abs_dalpha_per_row=delta)
    runner.close()
    res["config2"] = cfg2

    # ---- config 4's ICP arm and the large batch: Philox coin ----
    def batch(k, C):
        m = models[k]
        th = np.zeros((C, m.K + 10)); th[:, 0] = 1.0
        th[:, 10:] = np.random.default_rng(4).normal(0, 1.0, (C, m.K))     # random inits
        r = core.StdIcp(m, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=C)
        out, ms, wall, launches = _timed(r, th, (1e-15,), ITERS - 1, a.repeats, seed=7)
        r.close()
        return dict(K=m.K, fits=C, iterations=ITERS, device_ms=ms, fits_per_s=C / (ms * 1e-3),
                    fit_iterations_per_s=C * ITERS / (ms * 1e-3), cp_queries_per_s=C * ITERS * N / (ms * 1e-3),
                    launches_per_iteration=launches / ITERS, wall_ms=wall * 1e3, failed_fits=int((out["status"] != 0).sum()),
                    target_sampling_share=float(out["log_direction"].mean()))

    res["config4_icp_arm"] = [batch("100", 100), batch("200", 100)]
    res["fits_2368"] = batch("100", 2368)
    res["config4_icp_arm_targets"] = targets_section(ctx, fx, models, ids, [int(g) for g in a.groups.split(",")], a.repeats)
    for m in models.values():
        m.close()
    tgt.close(); ctx.close()
    s = json.dumps(res)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
