"""MCMC samples/s of the fused runner against the number of chains (config-1 workload), with and without the rejection
look-ahead: where the batch stops being latency-bound. SCHEDULES=auto,eager,lazy also times the step-by-step runner (W = 0)
under each posterior schedule (icp_debug_chain_schedule)."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from icp_proposal_b200 import _lib, core  # noqa: E402

m, tv, tc, ids, eids, tp = bench.workload()
ctx = core.Context(0)
model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
tgt = core.Target(ctx, tv, tc)
dev = torch.device("cuda", 0)
ru = _lib.RANK_UPDATE_INT8
pt = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, rank_update=ru)
pm = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=ru)
comps = [dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pt), dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pm),
         dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
widths = [int(w) for w in os.environ.get("WIDTHS", "0,2,4,8").split(",")]
schedules = os.environ.get("SCHEDULES", "auto").split(",")
out = {}
for C in [int(c) for c in os.environ.get("CHAINS", "1,8,16,32,64,148,296,592,1184,2368").split(",")]:
    th0 = torch.from_numpy(bench.init_thetas(m, C + 1)[1:].copy()).to(dev)
    for W, sch in [(w, x) for w in widths for x in schedules if w == 0 or x == "auto"]:
        if C * max(W, 1) > 4736:
            continue
        chain = core.Chain(model, tgt, comps, ev, max_chains=C)
        chain.set_lookahead(W)
        chain.schedule(sch)
        steps = 400 if C <= 592 else 100
        chain.run_device(C, 300, th0.data_ptr(), seed=1024)     # burn-in
        chain.run_device(C, steps, None, seed=1024)
        ms, _ = chain.last_run_stats()
        r = chain.last_run_rounds()
        key = f"C{C}_W{W}" + ("" if sch == "auto" else "_" + sch)
        out[key] = {"samples_per_s": C * steps / (ms * 1e-3), "ms_per_step": ms / steps, "ms_per_round": ms / r, "steps_per_round": steps / r}
        print(f"C {C:5d} W {W:2d} {sch:5s} {C * steps / (ms * 1e-3):12.0f} samples/s  {ms / steps:.4f} ms/step  {ms / r:.4f} ms/round  {steps / r:.2f} steps/round", flush=True)
        chain.close()
print(json.dumps(out))
