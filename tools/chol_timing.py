"""Phase times inside k_cholesky_packed from clock64() stamps of thread 0 (experiment build only).
    ICPCUDA_LIB_TAG=timing ICPCUDA_NVCC_EXTRA=-DICP_FUSED_TIMING python icp-proposal_b200/build.py
    ICPCUDA_LIB_TAG=timing python tools/chol_timing.py [--chains 2368] [--whitened]
The default table is the per-call posterior (icp_posterior, mu form). --whitened also factorises the same matrices in both
forms through icp_debug_factor: the mu form and the chain runner's form (y = L^-1 b in the mean slot, no back substitution).
"""
import argparse
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from icp_proposal_b200 import _lib, core  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--chains", type=int, default=2368)
ap.add_argument("--whitened", action="store_true")
a = ap.parse_args()
m, tv, tc, ids, eids, tp = bench.workload()
ctx = core.Context(0)
model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
tgt = core.Target(ctx, tv, tc)
prop = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, 1, True, ids, tp, rank_update=_lib.RANK_UPDATE_INT8)
th = bench.init_thetas(m, a.chains)
prop.posterior(th, want_M=False)
th2 = th.copy(); th2[:, 10:] += 1e-3
lib = _lib.load()
n = min(a.chains, 8192)
lib.icp_debug_fused_timing.argtypes = [C.c_void_p, C.c_int]
names = {8: "load M, b", 9: "factorisation (all 13 block columns)", 1: "  warp 0: column update (diagonal block + rhs)", 2: "  warp 0: 8 x 8 diagonal factor",
         3: "  barrier after update / diagonal", 4: "  panel solve", 5: "  barrier after the panel", 10: "back substitution",
         11: "store L, mean, quadratic form"}


def table(title):
    buf = np.zeros(12 * n, np.int64)
    assert lib.icp_debug_fused_timing(buf.ctypes.data, 12 * n) == 0
    t = buf.reshape(n, 12)
    print(f"k_cholesky_packed, {title}, {n} CTAs: median clocks of thread 0 (p10 .. p90)")
    for k, nm in names.items():
        v = t[:, k]
        print(f"  {nm:48s} {np.median(v):9.0f}  ({np.percentile(v, 10):.0f} .. {np.percentile(v, 90):.0f})")
    tot = np.median(t[:, 8] + t[:, 9] + t[:, 10] + t[:, 11])
    print(f"  {'total (median of the per-CTA sum)':48s} {tot:9.0f}")


if a.whitened:
    mu, M, _ = prop.posterior(th2, want_M=True)
    b = np.einsum("cij,cj->ci", M, mu)
    to = th2.copy(); to[:, 10:] += 1e-2
    for ymean in (False, True):
        for _ in range(2):   # the second launch is the one read back (modules loaded, L2 in the same state for both forms)
            ctx.factor(M, b, th2, to, 0.1, ymean=ymean)
        table("chain runner form (mean slot y = L^-1 b)" if ymean else "mu form")
else:
    prop.posterior(th2, want_M=False)
    table("per-call posterior (mu form)")
