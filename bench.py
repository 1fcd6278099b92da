#!/usr/bin/env python
"""bench.py - MCMC samples/sec (femur GPMM-100 shape) and closest-point queries/sec on B200.

One "step" is one Metropolis-Hastings step of every chain resident on the GPU (C samples per step and
GPU). Workload = BASELINE.json configs[2]/[3] shape: synthetic femur twin (N=1622, T=3240, K=101),
the config-1 proposal mixture 0.9*(0.5 ICP target-sampling + 0.5 ICP model-sampling, n=2K) + 0.1*RW(0.1)
and the prior x Gaussian-point(sd 2, 4K points, model->target) evaluator
(apps/femur/IcpProposalRegistration.scala:59-61,70-72,85), C independent random-init chains batched per
GPU (apps/femur/RunMHRandomInitComparison.scala shape; init alpha ~ N(0, 0.1 I) as
apps/femur/RandomSamplesFromModel.scala:28-36). Chains shard over GPUs with no data-path collective
(weak scaling: C chains per GPU); NCCL only gathers the chain statistics at the end.

    python bench.py --gpus N --steps K --warmup W          # this framework (libicpcuda.so)
    python bench.py --impl reference ...                    # the CPU path (oracle port) on the host cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mcmc_samples_per_sec_femur_gpmm100"
UNIT = "samples/s"
K_RANK = 101


def workload():
    from icp_proposal_b200 import synth
    m = synth.femur_twin(rank=K_RANK)
    tv, tc, _ = synth.synthetic_target(m, seed=7, alpha_sd=0.5)
    K = K_RANK
    ids = np.arange(2 * K, dtype=np.int32)               # first n vertices (SURVEY Appendix B1)
    eids = np.arange(4 * K, dtype=np.int32)
    tp = tv[:: max(1, len(tv) // (2 * K))][: 2 * K].copy()  # stand-in for VTK-decimated target points
    return m, tv, tc, ids, eids, tp


def init_thetas(m, n, offset=0):
    K = K_RANK
    th = np.zeros((n, K + 10))
    th[:, 0] = 1.0
    th[:, 7:10] = m["ref"].mean(0)
    for i in range(n):
        g = offset + i
        if g > 0:   # RandomSamplesFromModel.scala:28-36: index 0 starts from the mean, the others from N(0, 0.1 I)
            th[i, 10:] = np.random.default_rng(1024 + g).normal(0.0, np.sqrt(0.1), K)
    return th


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout.readlines()), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
def oracle_chain_rate(m, tv, tc, ids, eids, tp, n_chains, n_steps, threads, closed_form, first_chain=0):
    """Times the CPU restatement (oracle port) of the same chain on the host cores."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as orc

    K = K_RANK
    th0 = init_thetas(m, n_chains, first_chain)

    def one(c):
        om = orc.Model(m["ref"], m["cells"], m["basis"], m["variance"])   # per thread: the caches are not shared
        ot = orc.Mesh(tv, tc)
        pt = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, 1, True, ids, tp)
        pm = orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, 0, True, ids, tp)
        comps = [dict(kind=0, weight=0.45, icp=pt), dict(kind=0, weight=0.45, icp=pm), dict(kind=1, weight=0.1, sd=0.1)]
        rng = np.random.default_rng(99 + c)
        r = orc.chain_run(om, ot, comps, True, orc.EVAL_INDEPENDENT, 0, (0.0, 2.0), eids, tp, th0[c], n_steps,
                          rng.random(n_steps), rng.normal(size=(n_steps, K)), rng.random(n_steps), closed_form=closed_form)
        return r["n_accepted"]

    orc.lib()
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        acc = list(ex.map(one, range(n_chains)))
    dt = time.perf_counter() - t0
    return n_chains * n_steps / dt, dt, float(np.sum(acc)) / (n_chains * n_steps)


def enable_cpu_blas():
    """The timed CPU arm runs its dense linear algebra on the box's OpenBLAS / LAPACK (as Breeze does through netlib-java
    when a native BLAS is present); returns a short description for the JSON line."""
    from oracle import oracle as orc
    path = orc.use_blas(True)
    return ("OpenBLAS dgemm/dgemv + LAPACKE dsyevd, 1 BLAS thread per chain (%s)" % os.path.basename(path)) if path else \
        "built-in C loops (no OpenBLAS found on this box)"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    m, tv, tc, ids, eids, tp = workload()
    blas = enable_cpu_blas()
    cores = os.cpu_count() or 1
    threads = max(1, min(cores, 32))
    per = max(1, args.ref_steps)
    rates = []
    t_all = time.perf_counter()
    for s in range(args.warmup + args.steps):
        rate, dt, acc = oracle_chain_rate(m, tv, tc, ids, eids, tp, threads, per, threads, closed_form=False, first_chain=s * threads)
        if s >= args.warmup:
            rates.append((rate, dt))
    value = float(np.mean([r for r, _ in rates]))
    ms = float(np.mean([d for _, d in rates]) * 1e3)
    sample = (f"{threads} chains x {per} MH steps per bench step on {threads} threads (1 core per chain, reference structure: "
              f"SVD-rotated basis + full-mesh regressions; linear algebra: {blas})")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "femur GPMM-100 twin (N=1622,T=3240,K=101), config-1 ICP mixture + Gaussian-point evaluator, independent chains",
                       "chains": threads, "n_icp_points": int(len(ids)), "n_eval_points": int(len(eids))},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample, "linear_algebra": blas},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "wall_s": time.perf_counter() - t_all}
    emit(line)


def profile_constants():
    """DRAM traffic per launch and lane utilisation are ncu counters: they cannot be measured inside a timed run. They are
    read from the committed digest of the latest ncu --set full capture (profiles/traffic.json, written by
    tools/ncu_traffic.py from the .ncu-rep) and labelled as profile constants in the JSON line."""
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
        return json.load(f)


def per_call_latency(m, model, pt, pm, ev, th0_host, iters=40):
    """The literal drop-in path: one MH step as a stock Scalismo chain drives it through the per-call entry points
    (icp_propose, icp_log_transition both ways for both ICP components, icp_eval_log_value), one chain per host thread on
    SHARED proposal / evaluator handles (RunMHRandomInitComparison.scala:59-86 uses 10 threads). Steps/s whole job."""
    from concurrent.futures import ThreadPoolExecutor

    K = K_RANK

    def chain(t, n):
        rng = np.random.default_rng(500 + t)
        th = th0_host[t % len(th0_host)].copy()[None]
        for _ in range(n):
            z = rng.normal(size=(1, K))
            prop = (pt if rng.random() < 0.5 else pm).propose(th, z)
            for p in (pt, pm):
                p.log_transition(th, prop)
                p.log_transition(prop, th)
            ev.log_value(prop)
            th = prop           # always move on: every step needs fresh posteriors, as an accepted step does
        return n

    out = {}
    chain(0, 5)                 # warm-up: sizes the handles' scratch
    with ThreadPoolExecutor(max_workers=10) as ex:   # ... and that of the call slots concurrent calls on a handle lease
        list(ex.map(lambda t: chain(t, 5), range(10)))
    for threads in (1, 10):
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=threads) as ex:
            done = sum(ex.map(lambda t: chain(t, iters), range(threads)))
        dt = time.perf_counter() - t0
        out[f"threads_{threads}"] = {"steps_per_s": done / dt, "ms_per_step_per_thread": dt / iters * 1e3}
    # the same MH step with C chains funnelled into ONE batched call per entry point (SURVEY 8b: "better: the Scala side
    # funnels the C chains into one batched call"): whole-job steps/s = C x calls/s
    for Cb in (10, 100):
        rng = np.random.default_rng(900 + Cb)
        th = th0_host[:Cb].copy()
        n = max(10, iters // 2)
        t0 = None
        for k in range(n + 2):
            if k == 2:          # two untimed steps: the first sizes the scratch for this batch, the second captures the graphs
                t0 = time.perf_counter()
            z = rng.normal(size=(Cb, K))
            prop = (pt if rng.random() < 0.5 else pm).propose(th, z)
            for p in (pt, pm):
                p.log_transition(th, prop)
                p.log_transition(prop, th)
            ev.log_value(prop)
            th = prop
        dt = time.perf_counter() - t0
        out[f"batched_{Cb}_chains_per_call"] = {"steps_per_s": Cb * n / dt, "ms_per_batched_step": dt / n * 1e3}
    out["note"] = ("per-call C ABI, C = 1 per call, host buffers in and out on every call; 7 calls per MH step "
                   "(1 propose, 4 log_transition, 1 eval + the posterior cache); the threads share ONE target-sampling proposal, ONE "
                   "model-sampling proposal and ONE evaluator handle like the reference's fitting threads "
                   "(RunMHRandomInitComparison.scala:59-86); concurrent calls on a handle run on the handle's pool of call "
                   "slots (own stream and scratch each) and share its posterior cache")
    return out


DUMP_LIMIT_BYTES = 60 << 20     # with the .npy headers, under 64 MB


def dump_outputs(out_dir, arrays):
    """Writes what the timed run returned for its last step, one row per chain, as <out_dir>/<name>.npy in float64, so that
    two builds can be compared output for output. Above DUMP_LIMIT_BYTES a fixed seeded sample of the chains is written;
    chain.npy holds the indices of the chains written."""
    arrays = {k: v.cpu().numpy().reshape(v.shape[0], -1).astype(np.float64) for k, v in arrays.items()}
    n = len(next(iter(arrays.values())))
    per_chain = 8 * (1 + sum(a.shape[1] for a in arrays.values()))
    chain = np.arange(n)
    if n * per_chain > DUMP_LIMIT_BYTES:
        chain = np.sort(np.random.default_rng(0).choice(n, DUMP_LIMIT_BYTES // per_chain, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "chain.npy"), chain.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[chain].squeeze(1) if a.shape[1] == 1 else a[chain])


# ---------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from icp_proposal_b200 import _lib, core, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG"):
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries exactly one JSON line
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    m, tv, tc, ids, eids, tp = workload()
    K, L = K_RANK, K_RANK + 10
    C = args.chains
    ctx = core.Context(local)
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, tv, tc)
    # rank update of the ICP posteriors: INT8 tensor cores (tcgen05, split-integer emulation of the FP64 product, 1e-8 on the
    # posterior mean against the 1e-5 contract) by default; --rank-update fp64 selects the FP64 tensor pipe (DMMA, 1e-12)
    ru = _lib.RANK_UPDATE_INT8 if args.rank_update == "int8" else _lib.RANK_UPDATE_FP64
    pt = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, rank_update=ru)
    pm = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=ru)
    comps = [dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pt), dict(kind=_lib.PROP_ICP, weight=0.45, proposal=pm),
             dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
    chain = core.Chain(model, tgt, comps, ev, max_chains=C)
    th0_host = init_thetas(m, C, rank * C)

    # ---- device-resident arm ("value"): theta0 and the chain log live in HBM ---------------------------------
    steps, warm = args.steps, args.warmup
    th0 = torch.from_numpy(th0_host).to(dev)
    log_comp = torch.empty((steps, C), dtype=torch.int32, device=dev)
    log_acc = torch.empty((steps, C), dtype=torch.uint8, device=dev)
    log_val = torch.empty((steps, C, 3), dtype=torch.float64, device=dev)
    log_th = torch.empty((steps, C, L), dtype=torch.float64, device=dev)
    th_final = torch.empty((C, L), dtype=torch.float64, device=dev)
    n_acc = torch.zeros(C, dtype=torch.int64, device=dev)
    torch.cuda.synchronize()
    seed, off = 1024, rank * C
    chain.run_device(C, warm, th0.data_ptr(), seed=seed, chain_id_offset=off)       # W warm-up steps (+ state of theta0)
    with ClockSampler(local) as clocks:
        barrier()
        t0 = time.perf_counter()
        chain.run_device(C, steps, None, seed=seed, chain_id_offset=off, log_component=log_comp.data_ptr(),
                         log_accepted=log_acc.data_ptr(), log_values=log_val.data_ptr(), log_theta=log_th.data_ptr(),
                         theta_final=th_final.data_ptr(), n_accepted=n_acc.data_ptr())   # exactly K steps, resumed
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
    dev_ms, launches = chain.last_run_stats()       # CUDA events on the library stream around the K steps
    t_ms = max_over_ranks(dev_ms)
    value = world * C * steps / (t_ms * 1e-3)
    accept_rate = float(log_acc.float().mean().item())
    if args.dump_outputs and rank == 0:     # rank 0 runs the same chains at any --gpus
        dump_outputs(args.dump_outputs, {"component": log_comp[-1], "accepted": log_acc[-1], "values": log_val[-1],
                                         "theta": log_th[-1], "theta_final": th_final, "n_accepted": n_acc})

    # ---- sustained arm: >= 2000 resumed steps of the same chains (seconds under load, clocks sampled) -------
    sustained = None
    if args.sustain_steps > 0:
        S = args.sustain_steps
        s_comp = torch.empty((S, C), dtype=torch.int32, device=dev); s_acc = torch.empty((S, C), dtype=torch.uint8, device=dev)
        s_val = torch.empty((S, C, 3), dtype=torch.float64, device=dev); s_th = torch.empty((S, C, L), dtype=torch.float64, device=dev)
        torch.cuda.synchronize()
        with ClockSampler(local) as sclocks:
            barrier()
            chain.run_device(C, S, None, seed=seed, chain_id_offset=off, log_component=s_comp.data_ptr(),
                             log_accepted=s_acc.data_ptr(), log_values=s_val.data_ptr(), log_theta=s_th.data_ptr())
            barrier()
        s_ms, _ = chain.last_run_stats()
        s_ms = max_over_ranks(s_ms)
        sustained = {"value": world * C * S / (s_ms * 1e-3), "unit": UNIT, "steps": S, "ms_per_step": s_ms / S, "seconds": s_ms * 1e-3,
                     "accept_rate": float(s_acc.float().mean().item()), "clocks": sclocks.summary(),
                     "note": "the same chains resumed for S more steps with the full chain log written to HBM (%.1f GB)" %
                             ((s_comp.nbytes + s_acc.nbytes + s_val.nbytes + s_th.nbytes) / 1e9)}
        del s_comp, s_acc, s_val, s_th

    # ---- the same K steps with the other arithmetic of the rank update (comparison only) --------------------------------
    other = None
    if rank == 0 and world == 1:
        oru = _lib.RANK_UPDATE_FP64 if ru == _lib.RANK_UPDATE_INT8 else _lib.RANK_UPDATE_INT8
        opt_ = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, rank_update=oru)
        opm_ = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=oru)
        ocomps = [dict(kind=_lib.PROP_ICP, weight=0.45, proposal=opt_), dict(kind=_lib.PROP_ICP, weight=0.45, proposal=opm_),
                  dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.1, sd=0.1)]
        ochain = core.Chain(model, tgt, ocomps, ev, max_chains=C)
        o_th = torch.empty((steps, C, L), dtype=torch.float64, device=dev); o_acc = torch.empty((steps, C), dtype=torch.uint8, device=dev)
        ochain.run_device(C, warm, th0.data_ptr(), seed=seed, chain_id_offset=off)
        torch.cuda.synchronize()
        ochain.run_device(C, steps, None, seed=seed, chain_id_offset=off, log_accepted=o_acc.data_ptr(), log_theta=o_th.data_ptr())
        torch.cuda.synchronize()
        o_ms, _ = ochain.last_run_stats()
        same = (o_acc == log_acc)
        # chains whose accept decisions all agree took the same path: their states differ by the arithmetic alone
        agree = same.all(dim=0)
        dth = (o_th - log_th).abs().amax(dim=2)[:, agree]
        scale = log_th.abs().amax().item()
        other = {"rank_update": "fp64" if oru == _lib.RANK_UPDATE_FP64 else "int8", "value": C * steps / (o_ms * 1e-3), "unit": UNIT,
                 "ms_per_step": o_ms / steps, "accept_decisions_equal": float(same.float().mean().item()),
                 "chains_with_identical_decisions": int(agree.sum().item()),
                 "max_abs_theta_diff_on_those": float(dth.max().item()) if dth.numel() else None, "theta_scale": scale,
                 "note": "same seed, same chains, the other arithmetic of the rank update; states compared after every one of the K steps"}
        del o_th, o_acc
        ochain.close(); opt_.close(); opm_.close()

    # ---- end-of-run exchange through the library's own NCCL entry points (icp_comm_*; the only collectives, not on the
    # per-sample path): all-gather of the FULL chain logs of the timed steps and all-reduce of the posterior variability
    # maps over the final states. torch.distributed only ferries the 128-byte communicator id. ---------------------------
    gather_ms = None
    gather = None
    if world > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid = torch.from_numpy(core.Comm.unique_id(ctx)).to(dev)
        dist.broadcast(uid, 0)
        comm = core.Comm(ctx, rank, world, uid.cpu().numpy())
        g_comp = torch.empty((world, steps, C), dtype=torch.int32, device=dev); g_acc = torch.empty((world, steps, C), dtype=torch.uint8, device=dev)
        g_val = torch.empty((world, steps, C, 3), dtype=torch.float64, device=dev); g_th = torch.empty((world, steps, C, L), dtype=torch.float64, device=dev)
        g_fin = torch.empty((world, C, L), dtype=torch.float64, device=dev); g_nacc = torch.empty((world, C), dtype=torch.int64, device=dev)
        lio, gio = _lib.ChainIO(), _lib.ChainIO()
        lio.log_component, lio.log_accepted, lio.log_values, lio.log_theta = log_comp.data_ptr(), log_acc.data_ptr(), log_val.data_ptr(), log_th.data_ptr()
        lio.theta_final, lio.n_accepted = th_final.data_ptr(), n_acc.data_ptr()
        gio.log_component, gio.log_accepted, gio.log_values, gio.log_theta = g_comp.data_ptr(), g_acc.data_ptr(), g_val.data_ptr(), g_th.data_ptr()
        gio.theta_final, gio.n_accepted = g_fin.data_ptr(), g_nacc.data_ptr()
        comm.chainlog_gather(steps, C, K, lio, gio)                       # warm-up (NCCL sets up its channels on first use)
        barrier()
        ms, nbytes = comm.chainlog_gather(steps, C, K, lio, gio)
        gather_ms = max_over_ranks(ms)
        ok = bool(torch.equal(g_th[rank], log_th) and torch.equal(g_acc[rank], log_acc))
        t0 = time.perf_counter()
        vmaps = comm.variability_allreduce(model, th_final[: min(C, 256)].cpu().numpy(), sum_normals=True)
        var_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
        gather = {"chainlog_gather_ms": gather_ms, "bytes_received_per_rank": int(nbytes), "GBps_per_rank": nbytes / (gather_ms * 1e-3) / 1e9,
                  "own_shard_intact": ok, "whole_job_accept_rate": float(g_acc.float().mean().item()),
                  "variability_allreduce_ms": var_ms, "variability_samples": int(vmaps["n"]),
                  "mean_total_variance": float(vmaps["total_variance"].mean()), "nccl_version": comm.nccl_version(),
                  "note": "icp_chainlog_gather (ncclAllGather of every log array of the timed steps, grouped) and "
                          "icp_variability_allreduce (two ncclAllReduce passes), both through libicpcuda's own communicator"}
        del g_comp, g_acc, g_val, g_th, g_fin, g_nacc
        comm.close()

    # ---- end-to-end arm: the public host-buffer call (pinned host memory in, chain log out) ---------------
    pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
    h_th0 = pin((C, L), torch.float64); h_th0[:] = th0_host
    e_steps = steps
    io = _lib.ChainIO()
    io.seed, io.chain_id_offset = seed, off
    h_comp, h_acc = pin((e_steps, C), torch.int32), pin((e_steps, C), torch.uint8)
    h_val, h_thl = pin((e_steps, C, 3), torch.float64), pin((e_steps, C, L), torch.float64)
    h_fin, h_nacc = pin((C, L), torch.float64), pin((C,), torch.int64)
    io.log_component, io.log_accepted, io.log_values, io.log_theta = (h_comp.ctypes.data, h_acc.ctypes.data, h_val.ctypes.data,
                                                                      h_thl.ctypes.data)
    io.theta_final, io.n_accepted = h_fin.ctypes.data, h_nacc.ctypes.data
    import ctypes as Cc
    # untimed warm-up call of the same size (sizes the library's staging buffers; W >= 3 steps run inside it too)
    _lib.check(chain.lib.icp_chain_run(chain.h, C, max(warm, e_steps), _lib.dptr(h_th0), Cc.byref(io)), ctx.h)
    e2e_runs = []
    for _ in range(5):          # five timed end-to-end calls of exactly K steps; the median is reported, all are listed
        barrier()
        t0 = time.perf_counter()
        _lib.check(chain.lib.icp_chain_run(chain.h, C, e_steps, _lib.dptr(h_th0), Cc.byref(io)), ctx.h)
        torch.cuda.synchronize()
        e2e_runs.append(max_over_ranks((time.perf_counter() - t0) * 1e3))
    e2e_ms = float(np.median(e2e_runs))
    barrier()
    # the host call evaluates theta0 once (1 extra state) before the K steps: count K steps of C samples
    e2e_value = world * C * e_steps / (e2e_ms * 1e-3)
    h2d = h_th0.nbytes / e_steps
    d2h = (h_comp.nbytes + h_acc.nbytes + h_val.nbytes + h_thl.nbytes + h_fin.nbytes + h_nacc.nbytes) / e_steps

    # ---- closest-point traversal on every GPU: 1000 B / query on the femur mesh (SURVEY 8d), 1e6 device-resident queries
    # per GPU (the target BVH is replicated, queries shard like chains); whole-job queries/s = the sum over the ranks -----
    import ctypes as Cc2
    cp = {}
    nq = 1_000_000
    for name, q in (("near_surface", synth.near_surface_queries(tv, tc, nq, seed=11 + 100 * rank)),
                    ("far_field", synth.far_field_queries(tv, nq, seed=12 + 100 * rank))):
        qd = torch.from_numpy(q).to(dev)
        tri = torch.empty(nq, dtype=torch.int32, device=dev); cpd = torch.empty((nq, 3), dtype=torch.float64, device=dev)
        d2 = torch.empty(nq, dtype=torch.float64, device=dev)
        ms = Cc2.c_double(0)
        barrier()
        _lib.check(chain.lib.icp_debug_time_closest_point(tgt.h, nq, qd.data_ptr(), tri.data_ptr(), cpd.data_ptr(), d2.data_ptr(),
                                                          10, Cc2.byref(ms)), ctx.h)
        worst = max_over_ranks(ms.value)     # device time of the slowest rank
        cp[name] = {"queries_per_s": world * nq / (worst * 1e-3), "queries_per_s_per_gpu": nq / (ms.value * 1e-3), "ms_per_launch": ms.value,
                    "algorithmic_GBps": nq * 1000.0 / (ms.value * 1e-3) / 1e9, "n_gpus": world}
        del qd, tri, cpd, d2

    line = None
    if rank == 0:
        l2_gbs = ctx.l2_bandwidth(32 << 20)     # L2 -> SM reads over an L2-resident 32 MB working set, measured live
        per_call = per_call_latency(m, model, pt, pm, ev, th0_host)
        # ---- per-kernel device times (CUDA events on the launching stream, eager pass over the same workload) --
        prof_steps = max(2, min(steps, 8))
        prof = chain.profile(th0_host, prof_steps, seed=seed)
        total_prof = sum(v["ms"] for v in prof.values()) or 1.0
        shares = {k: round(v["ms"] / total_prof, 4) for k, v in prof.items() if v["launches"]}
        fp64 = ctx.fp64_peak()
        peaks, peak_src = measured_peaks()
        prof_const = profile_constants()
        # posterior = rank-update kernel (k_posterior_fused<.., CHOL = false>: M = I + A^T A, b = A^T y on the FP64 tensor
        # pipe) + k_cholesky_packed; each twice per step (target- and model-sampling proposal). The rank update dominates.
        # Its algorithmic flops per chain-posterior (SURVEY 8d): 2*3n*K^2 (M) + 2*3n*K*3 (Sigma^-1 apply) = 12.4 MFLOP at
        # n = 202, K = 101 - what the reference's regression computes per posterior before it factorises.
        n_obs = len(ids)
        flops_post = 2.0 * 3 * n_obs * K * K + 2.0 * 3 * n_obs * K * 3
        flops_chol = K ** 3 / 3.0 + 2.0 * K * K
        # executed on the tensor pipe: only the 91 lower-triangle 8x8 blocks (Kp = 104), and one row per observation instead
        # of three for the model-sampling proposal (constant-Gram fast path); Cholesky as above
        nb = (K + 7) // 8
        blocks = nb * (nb + 1) // 2
        rows_t, rows_m = 3 * 8 * ((n_obs + 7) // 8), 24 * ((n_obs + 23) // 24)
        flops_exec = 0.5 * (2.0 * 64 * blocks * rows_t + 2.0 * 64 * blocks * rows_m)
        Kp = 8 * nb
        ch = prof.get("cholesky_solve", {"ms": 0.0, "launches": 0})
        ch_ms = ch["ms"] / max(ch["launches"], 1)
        # k_cholesky_packed per launch: reads the packed blocks + b, writes the lower triangle of L + mu
        ch_bytes = C * 8.0 * (64 * blocks + Kp + Kp * (Kp + 1) / 2 + Kp)
        roof_chol = None
        if ch["launches"]:
            roof_chol = {"bound": "hbm", "kernel": "k_cholesky_packed", "achieved": ch_bytes / (ch_ms * 1e-3) / 1e9,
                         "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ch_bytes / (ch_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "traffic": prof_const["cholesky"]["dram_bytes_per_launch"] * C / prof_const["cholesky"]["chains"],
                         "traffic_source": prof_const["cholesky"]["source"] + " (profile constant, scaled by C)",
                         "avg_launch_ms": ch_ms, "flops_per_launch": flops_chol * C,
                         "share_of_step": shares.get("cholesky_solve"),
                         "note": "a chain of Kp dependent pivots per matrix: latency-bound by construction (4 chains per SM hide "
                                 "it); traffic = dram read + write per launch from profiles/r1j (ncu --set full, C = 2368), scaled by C"}
        pb = prof["posterior_build"]
        pb_ms = pb["ms"] / max(pb["launches"], 1)
        pb_tflops = flops_post * C / (pb_ms * 1e-3) / 1e12 if pb_ms > 0 else 0.0
        pb_hw = flops_exec * C / (pb_ms * 1e-3) / 1e12 if pb_ms > 0 else 0.0
        top = max(shares, key=shares.get)
        cpq = prof["closest_point_static"]
        cp_ms = cpq["ms"] / max(cpq["launches"], 1)
        roof_cp = {"bound": "l2", "kernel": prof_const["closest_point"]["kernel"] + " (1e6 near-surface queries, timed alone)",
                   "achieved": cp["near_surface"]["algorithmic_GBps"], "peak": l2_gbs, "unit": "GB/s",
                   "frac": cp["near_surface"]["algorithmic_GBps"] / l2_gbs if l2_gbs else None,
                   "peak_source": "L2 -> SM read bandwidth over an L2-resident 32 MB working set, measured live (icp_debug_l2_bandwidth); "
                                  "the tree + triangles (0.5 MB) are cache resident, so L2 - not HBM - is the ceiling (SURVEY 8d)",
                   "frac_of_hbm_copy": cp["near_surface"]["algorithmic_GBps"] / peaks["hbm_gbs"], "hbm_peak": peaks["hbm_gbs"],
                   "hbm_peak_source": peak_src, "bytes_per_query": 1000,
                   "traffic": prof_const["closest_point"]["dram_bytes_per_launch"],
                   "traffic_source": prof_const["closest_point"]["source"] + " (a PROFILE CONSTANT read from profiles/, not measured in this run)",
                   "lanes_active_per_instruction": prof_const["closest_point"].get("lanes_active_per_instruction"),
                   "far_field_frac": cp["far_field"]["algorithmic_GBps"] / l2_gbs if l2_gbs else None}
        roofline = {"bound": "tensor", "pipe": "FP64 tensor pipe (mma.sync.m8n8k4.f64, SASS DMMA)",
                    "kernel": "k_posterior_fused<.., CHOL = false> (rank update M = I + A^T A, b = A^T y)",
                    # frac = flops the kernel EXECUTES / measured DMMA peak: a hardware fraction (<= 1). The algorithmic figure
                    # of SURVEY 8d (what the reference's regression computes per posterior) is 2.6x the executed one because
                    # the kernel only forms the lower-triangle blocks and, on the constant-Gram path, one row per observation;
                    # it is reported as achieved_algorithmic / frac_algorithmic and may exceed 1.
                    "achieved": pb_hw, "peak": fp64["dmma_tflops"], "unit": "TFLOP/s",
                    "frac": pb_hw / fp64["dmma_tflops"] if fp64["dmma_tflops"] else None,
                    "achieved_algorithmic": pb_tflops,
                    "frac_algorithmic": pb_tflops / fp64["dmma_tflops"] if fp64["dmma_tflops"] else None,
                    "traffic": prof_const["rank_update"]["dram_bytes_per_launch"] * C / prof_const["rank_update"]["chains"],
                    "traffic_source": prof_const["rank_update"]["source"] + " (a PROFILE CONSTANT read from profiles/, scaled by C; not measured in this run)",
                    "traffic_note": "algorithmic bytes per launch = C * (8 * 64 * 91 + 8 Kp) written (packed M, b) ~ 112 MB plus the "
                                    "observation frames read (~ 48 MB); the basis rows come from L2",
                    "peak_source": "DMMA m8n8k4 micro-benchmark run live on this GPU (MEASURED_PEAKS.json has no FP64 figure); "
                                   "DFMA measured %.1f TFLOP/s" % fp64["dfma_tflops"],
                    "flops_per_launch": flops_post * C, "executed_flops_per_launch": flops_exec * C, "avg_launch_ms": pb_ms,
                    "share_of_step": shares.get("posterior_build"), "top_kernel_by_time": top,
                    "note": "achieved / frac count the flops actually executed (symmetry + constant Gram term exploited); "
                            "*_algorithmic count the reference's flops per posterior (SURVEY 8d)"}
        if ru == _lib.RANK_UPDATE_INT8:
            i8_peak = ctx.i8_peak()
            # executed on the INT8 tensor cores per chain-posterior: ceil(n / 32) steps x (3 | 1) K blocks of 32 rows x ten digit
            # pair products of 128 x 112 x 32 (issued as four 128 x 224 and two 128 x 112 MMAs)
            nst = (n_obs + 31) // 32
            ops_exec = 0.5 * (3 + 1) * nst * 10 * 2.0 * 128 * 112 * 32
            i8_hw = ops_exec * C / (pb_ms * 1e-3) / 1e12 if pb_ms > 0 else 0.0
            roofline = {"bound": "tensor", "pipe": "5th-generation tensor cores: tcgen05.mma kind::i8, INT32 accumulators in TMEM (SASS UTCIMMA / LDTM)",
                        "kernel": "k_rank_update_i8<3|1> (rank update M = I + A^T A, b = A^T y by split-integer emulation of the FP64 product: "
                                  "four balanced base-256 digits, ten digit-pair products, exact INT32 accumulation)",
                        "achieved": i8_hw, "peak": i8_peak, "unit": "TFLOP/s",
                        "frac": i8_hw / i8_peak if i8_peak else None,
                        "achieved_algorithmic": pb_tflops,
                        "frac_algorithmic_of_fp64_tensor_peak": pb_tflops / fp64["dmma_tflops"] if fp64["dmma_tflops"] else None,
                        "peak_bf16_dense_measured": peaks.get("bf16_tflops") or peaks.get("bf16_dense_tflops"),
                        "traffic": prof_const["rank_update_i8"]["dram_bytes_per_launch"] * C / prof_const["rank_update_i8"]["chains"],
                        "traffic_source": prof_const["rank_update_i8"]["source"] + " (a PROFILE CONSTANT read from profiles/, scaled by C; not measured in this run)",
                        "traffic_note": "algorithmic bytes per launch = C * (8 * 64 * 91 + 8 Kp) written (packed M, b) ~ 112 MB plus the "
                                        "observation frames read (~ 48 MB); the basis rows (1.2 GB per launch) come from L2",
                        "peak_source": "INT8 tensor-core rate of the same MMA tile (128 x 112 x 32, operands in shared memory) measured live on this "
                                       "GPU with 2 CTAs / SM (icp_debug_i8_gram); MEASURED_PEAKS.json holds bf16, not INT8; achieved / peak are "
                                       "integer tera-operations per second",
                        "flops_per_launch": flops_post * C, "executed_int8_ops_per_launch": ops_exec * C, "avg_launch_ms": pb_ms,
                        "share_of_step": shares.get("posterior_build"), "top_kernel_by_time": top,
                        "note": "achieved / frac count the INT8 operations the tensor cores execute (ten digit pairs of the full 128 x 112 tile); "
                                "achieved_algorithmic counts the reference's FP64 flops per posterior (SURVEY 8d). The kernel is bound by "
                                "the FP64 whitening + digit extraction in its converter warps and by shared-memory bandwidth (staging ring + "
                                "MMA operands), not by the tensor pipe: profiles/r2_i8_rank_update.md"}
        # ---- BASELINE.json configs[0] shape: ONE chain, fixed seed - latency-bound by construction (SURVEY 8d): steps/s of
        # the device-resident loop with a single resident chain, next to the 1-core CPU port below -------------------
        # The fused runner's rejection look-ahead (icp_chain_set_lookahead; automatic for <= 8 chains) evaluates the proposals of
        # the next 8 steps from the same state in one batched round - same chain log, 2.4 x fewer rounds at this acceptance rate.
        # th0_host[1] is a random-init chain (index 0 starts from the mean); 500 burn-in steps first, acceptance is high at first.
        sc_steps = 2000
        th1 = torch.from_numpy(np.ascontiguousarray(th0_host[1:2])).to(dev)
        single_chain = {}
        for name, width in (("step_by_step", 0), ("lookahead", -1)):
            chain.set_lookahead(width)
            sc_acc = torch.zeros(1, dtype=torch.int64, device=dev)
            chain.run_device(1, 500, th1.data_ptr(), seed=seed, chain_id_offset=off + 1)   # burn-in; sizes + captures the graph
            torch.cuda.synchronize()
            chain.run_device(1, sc_steps, None, seed=seed, chain_id_offset=off + 1, n_accepted=sc_acc.data_ptr())   # resumed
            sc_ms, _ = chain.last_run_stats()
            rounds = chain.last_run_rounds()
            single_chain[name] = {"steps_per_s": sc_steps / (sc_ms * 1e-3), "ms_per_step": sc_ms / sc_steps, "steps": sc_steps,
                                  "rounds": int(rounds), "accepted_total": int(sc_acc.item())}
        chain.set_lookahead(-1)
        single_chain.update(single_chain["lookahead"])
        single_chain["note"] = ("one chain resident on the GPU (configs[0] shape): every kernel of a step runs a single CTA / a handful "
                                "of warps, so a step is launch + dependent-latency time. 'lookahead' (the default for <= 8 chains): 8 lanes "
                                "propose the next 8 steps from the current state in one batched round, the first accepting lane is the "
                                "chain's next state - the log is bit-identical to 'step_by_step' (tests/test_gpu_round2.py::"
                                "test_rejection_lookahead_is_bit_identical). n_accepted counts from the start of the chain (burn-in included)")
        # ---- CPU baseline: the oracle port of the same chain on this box's host cores (bounded sample) ------
        cores = os.cpu_count() or 1
        blas = enable_cpu_blas()
        cb_rate, cb_dt, _ = oracle_chain_rate(m, tv, tc, ids, eids, tp, 1, args.cpu_steps, 1, closed_form=False)
        opt_rate, opt_dt, _ = oracle_chain_rate(m, tv, tc, ids, eids, tp, 1, args.cpu_steps * 20, 1, closed_form=True)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warm,
                "ms_per_step": t_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64 (rank update of the posterior: INT8 tensor-core emulation of the FP64 product, 1e-8)" if ru == _lib.RANK_UPDATE_INT8 else "f64",
                "data": "synthetic",
                "config": {"workload": "femur GPMM-100 twin (N=1622,T=3240,K=101), config-1 ICP mixture (0.45 target-sampling + 0.45 "
                                       "model-sampling ICP n=202, 0.1 random walk) + prior x Gaussian-point(sd 2, 404 pts) evaluator, "
                                       "independent random-init chains batched per GPU",
                           "rank_update": args.rank_update, "chains_per_gpu": C, "samples_per_step": world * C, "n_icp_points": int(len(ids)), "n_eval_points": int(len(eids)),
                           "parallelism": f"chains sharded over {world} GPU(s), no data-path collective",
                           "l2_policy": "per-step working set (posteriors 4x%.0f MB + meshes) exceeds L2" % (C * 104 * 104 * 8 / 1e6)},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / e_steps,
                        "runs_ms": e2e_runs, "note": "median of 5 host-buffer icp_chain_run calls of K steps: pinned theta0 in, full chain log out"},
                "gpu_launches": int(launches), "wall_ms_per_step": wall_ms / steps, "accept_rate": accept_rate,
                "clocks": clocks.summary(), "roofline": roofline, "roofline_cholesky": roof_chol, "roofline_closest_point": roof_cp, "closest_point": cp,
                "kernel_shares": shares, "kernel_ms_per_step": {k: v["ms"] / prof_steps for k, v in prof.items() if v["launches"]},
                "fp64_peak": fp64, "l2_read_gbs": l2_gbs, "gather_ms": gather_ms, "gather": gather, "single_chain": single_chain,
                "sustained": sustained, "other_rank_update": other, "per_call_api": per_call,
                "cpu_baseline": {"value": cb_rate, "unit": UNIT, "cores": 1, "kind": "port",
                                 "sample": f"1 chain x {args.cpu_steps} MH steps of the same workload, oracle in the reference's structure, 1 thread ({cb_dt:.1f} s); host has {cores} cores",
                                 "linear_algebra": blas},
                "cpu_baseline_optimised": {"value": opt_rate, "unit": UNIT, "cores": 1, "kind": "port",
                                           "sample": f"1 chain x {args.cpu_steps * 20} steps, oracle with the same closed forms as the device ({opt_dt:.1f} s)"},
                "device": ctx.version()}
        emit(line)
    barrier()
    if world > 1:
        dist.destroy_process_group()


_JSON_OUT = None


def _claim_stdout():
    """stdout must carry exactly one JSON line: keep a private handle on it and point fd 1 at stderr, so that whatever a
    native library prints (NCCL writes its version banner to stdout) lands on stderr."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    _claim_stdout()
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=4736, help="chains per GPU (32 x 148 SMs; 2368 gives 4 %% less, profiles/r2_session3.md)")
    ap.add_argument("--cpu-steps", type=int, default=120, help="MH steps of the cpu_baseline sample")
    ap.add_argument("--sustain-steps", type=int, default=2000, help="steps of the sustained-load arm (0 = skip)")
    ap.add_argument("--rank-update", default="int8", choices=["int8", "fp64"],
                    help="arithmetic of the posterior's rank update: INT8 tensor cores (tcgen05; default) or the FP64 tensor pipe")
    ap.add_argument("--ref-steps", type=int, default=12, help="MH steps per chain and bench step of --impl reference")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--impl b200 only: write what the timed run returned for its last step (one row per chain) to "
                         "DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.warmup < 1:
        args.warmup = 1
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
