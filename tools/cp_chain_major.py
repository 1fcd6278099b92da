"""Lane activity and time of the per-chain closest-point queries (k_nearest) on the bench workload.
    ICPCUDA_LIB_TAG=timing ICPCUDA_NVCC_EXTRA=-DICP_CP_TIMING python icp-proposal_b200/build.py   # libicpcuda_timing.so
    ICPCUDA_LIB_TAG=timing python tools/cp_chain_major.py [--chains 4736] [--steps 8]   # counters (and times of that build)
    python tools/cp_chain_major.py [--chains 4736]                                      # times of the product build
Times: the evaluator alone (icp_eval_log_value, model -> target, 404 points per chain, host clock around the synchronous
call) and closest_point_static of the eager per-kernel pass of a chain run (what bench.py reports as
kernel_ms_per_step.closest_point_static). Counters (timing build only): warp and lane iterations of the descent phase and of
the leaf phase of every k_nearest launch, for one evaluator call and for a chain run of --steps steps from the bench's
initial states; lanes active per node visit = lane iterations / warp iterations.
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from icp_proposal_b200 import _lib, core  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--chains", type=int, default=4736)
ap.add_argument("--steps", type=int, default=8)
ap.add_argument("--reps", type=int, default=30)
ap.add_argument("--out", default=None, help="write the results as JSON to this file")
a = ap.parse_args()

m, tv, tc, ids, eids, tp = bench.workload()
K = bench.K_RANK
ctx = core.Context(0)
model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
tgt = core.Target(ctx, tv, tc)
ru = _lib.RANK_UPDATE_INT8
pt = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, rank_update=ru)
pm = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=ru)
comps = [dict(kind=0, weight=0.45, proposal=pt), dict(kind=0, weight=0.45, proposal=pm), dict(kind=1, weight=0.1, sd=0.1)]
ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
chain = core.Chain(model, tgt, comps, ev, max_chains=a.chains)
th0 = bench.init_thetas(m, a.chains)
lib = _lib.load()
counters = getattr(lib, "icp_debug_cp_counters", None)   # timing build only
res = {"chains": a.chains, "lib": os.path.basename(_lib.LIB_PATH)}

# evaluator alone: the first call builds its seeds, the timed ones start from them (as in a chain)
ev.log_value(th0)
ts = []
for _ in range(a.reps):
    t0 = time.perf_counter()
    ev.log_value(th0)
    ts.append((time.perf_counter() - t0) * 1e3)
res["evaluator_call_ms"] = {"median": float(np.median(ts)), "min": float(np.min(ts))}
prof = chain.profile(th0, a.steps, seed=1024)
cps = prof["closest_point_static"]
res["closest_point_static_ms_per_step"] = cps["ms"] / a.steps
res["closest_point_static_launches_per_step"] = cps["launches"] / a.steps
print(f"{a.chains} chains ({res['lib']}): evaluator call {res['evaluator_call_ms']['median']:.3f} ms (min "
      f"{res['evaluator_call_ms']['min']:.3f}); closest_point_static {res['closest_point_static_ms_per_step']:.3f} ms per step "
      f"({res['closest_point_static_launches_per_step']:.1f} launches, eager pass of {a.steps} steps)")

if counters is not None:
    counters.argtypes = [C.c_void_p, C.c_int32]
    buf = np.zeros(6, np.uint64)

    def read(reset):
        assert counters(buf.ctypes.data, int(reset)) == 0
        return buf.astype(np.float64).copy()

    def report(name, cnt):
        wd, ld, wl, ll, warps, live = cnt
        r = {"warps": int(warps), "queries": int(live), "lanes_per_node_visit": ld / wd, "lanes_per_leaf_test": ll / wl,
             "warp_descent_iterations_per_warp": wd / warps, "descent_iterations_per_query": ld / live,
             "warp_leaf_rounds_per_warp": wl / warps, "leaf_tests_per_query": ll / live}
        print(f"  {name}: {r['lanes_per_node_visit']:.1f} of 32 lanes active per node visit, {r['lanes_per_leaf_test']:.1f} per "
              f"leaf test; a warp runs {r['warp_descent_iterations_per_warp']:.1f} node-visit iterations where its average "
              f"query needs {r['descent_iterations_per_query']:.1f}, and {r['warp_leaf_rounds_per_warp']:.1f} leaf rounds for "
              f"{r['leaf_tests_per_query']:.1f} leaf tests ({int(live)} queries in {int(warps)} warps)")
        res[name] = r

    read(True)
    ev.log_value(th0)
    report("evaluator", read(True))
    chain.run(th0, a.steps, seed=1024, log_theta=False)
    report("chain_run", read(True))

if a.out:
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
