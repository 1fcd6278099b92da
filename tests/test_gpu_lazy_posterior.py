"""The lazy posterior schedule of the step-by-step chain runner (chain.cu, DESIGN.md section 5): every run is compared with the
eager schedule (icp_debug_chain_schedule), which factors both ICP posteriors of every proposal, bit for bit - the chain log,
the final state, the counters, the status words and the best sample. Also: the factorisations it makes against a host replay
of the log, a mixture that takes both the certified and the fallback branch, and the cases that keep the eager schedule."""
import numpy as np
import pytest

from icp_proposal_b200 import _lib, core, synth

pytestmark = pytest.mark.gpu

K = 101
KEYS = ("component", "accepted", "values", "theta", "theta_final", "n_accepted", "status", "theta_best", "value_best")


class Setup:
    """GPMM-100 femur twin, G targets, each with the bench mixture (0.45 target-sampling ICP, 0.45 model-sampling ICP, 0.1 random
    walk of std-dev sd) or an ICP-only mixture, and an evaluator."""

    def __init__(self, ctx, femur, G=1, rank_update=_lib.RANK_UPDATE_INT8, evaluator="independent", sd=0.1, icp_only=False):
        base = dict(ref=femur["ref"], cells=femur["cells"], **femur["gpmm_100"])
        self.model = core.Model(ctx, base["ref"], base["cells"], base["basis"], base["variance"])
        self.entries, self.handles = [], []
        ids, eids = np.arange(2 * K), np.arange(4 * K)
        for g in range(G):
            tv = synth.model_instance(base, np.random.default_rng(100 + g).normal(0, 1.0, K))
            tv = tv + np.random.default_rng(7 + g).normal(0, 0.5, tv.shape)
            tgt = core.Target(ctx, tv, base["cells"])
            tp = tv[:: len(tv) // (2 * K)][: 2 * K]
            mk = lambda d: core.IcpProposal(self.model, tgt, 0.1, 10.0, 5.0, d, True, ids, tp, rank_update=rank_update)
            pt, pm = mk(_lib.TARGET_SAMPLING), mk(_lib.MODEL_SAMPLING)
            comps = [dict(kind=0, weight=0.45, proposal=pt), dict(kind=0, weight=0.45, proposal=pm)]
            if icp_only:
                comps = [dict(kind=0, weight=0.5, proposal=pt), dict(kind=0, weight=0.5, proposal=pm)]
            else:
                comps.append(dict(kind=1, weight=0.1, sd=sd))
            if evaluator == "hausdorff":
                ev = core.Evaluator(self.model, tgt, _lib.EVAL_HAUSDORFF, 0, True, 100.0)
            else:
                ev = core.Evaluator(self.model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
            self.entries.append((tgt, comps, ev))
            self.handles += [ev, pt, pm, tgt]

    def chain(self, C):
        if len(self.entries) > 1:
            ch = core.Chain(self.model, targets=self.entries, max_chains=C)
        else:
            ch = core.Chain(self.model, *self.entries[0], C)
        ch.set_lookahead(0)
        return ch

    def theta0(self, C, seed):
        rng = np.random.default_rng(seed)
        return np.stack([self.model.theta()] + [self.model.theta(rng.normal(0, np.sqrt(0.1), K)) for _ in range(C - 1)])

    def close(self):
        for h in self.handles:
            h.close()
        self.model.close()


def _assert_equal(a, b, what):
    for k in KEYS:
        assert np.array_equal(a[k], b[k], equal_nan=True), f"{k} differs ({what})"


def _both(ch, run, mode="lazy"):
    """run() under the eager schedule, then under `mode` ("lazy" wherever it applies, "auto" the runner's choice):
    (eager result, result, lazy?, counters)."""
    ch.schedule("eager")
    want = run()
    lazy, cnt = ch.schedule()
    assert not lazy and cnt == [0, 0, 0]
    ch.schedule(mode)
    got = run()
    lazy, cnt = ch.schedule()
    return want, got, lazy, cnt


def _replay(comp, accepted, n_icp=2):
    """Factorisations of the rule "factor the current posterior of the picked ICP component when it is missing; an accepted
    step leaves none", replayed over a chain log (theta0's posteriors are factored with its evaluation)."""
    n, C = comp.shape
    valid = np.ones((C, n_icp), bool)
    total = 0
    for t in range(n):
        for c in range(C):
            i = comp[t, c]
            if i < n_icp and not valid[c, i]:
                valid[c, i] = True
                total += 1
            if accepted[t, c]:
                valid[c] = False
    return total


@pytest.mark.parametrize("mode", ["auto", "lazy"])
@pytest.mark.parametrize("rank_update", [_lib.RANK_UPDATE_INT8, _lib.RANK_UPDATE_FP64])
@pytest.mark.parametrize("C", [1, 32, 149, 300, 4736])
def test_bench_mixture_equals_eager_schedule(ctx, femur, rank_update, C, mode):
    """The bench mixture at GPMM-100: the runner chooses the lazy schedule from two chains per SM on (148 SMs); its log equals
    the eager one bit for bit, every step is certified (the random walk's density dominates), and its factorisations are the
    host replay's."""
    S = Setup(ctx, femur, rank_update=rank_update)
    n = 12 if C == 4736 else 24
    th0 = S.theta0(C, 5)
    ch = S.chain(C)
    want, got, lazy, cnt = _both(ch, lambda: ch.run(th0, n, seed=5), mode)
    _assert_equal(want, got, f"C = {C}")
    import torch
    assert lazy == (mode == "lazy" or C >= 2 * torch.cuda.get_device_properties(0).multi_processor_count)
    if not lazy:
        assert cnt == [0, 0, 0]
        ch.close(); S.close()
        return
    assert 0 < got["n_accepted"].sum() < C * n
    assert cnt[1] == 0 and cnt[2] == C * n
    assert cnt[0] == _replay(got["component"], got["accepted"])
    assert cnt[0] < C * n          # under the one factorisation per chain-step of either ICP component picked
    ch.close(); S.close()


@pytest.mark.parametrize("evaluator", ["independent", "hausdorff"])
def test_resume_statistics_and_targets(ctx, femur, evaluator):
    """A 3-target handle with statistics on, run 10 + 14 steps through the resumed device runner: the log and every chain's
    variability maps equal the eager schedule's; the resumed part keeps the schedule of the run it resumes."""
    import torch
    S = Setup(ctx, femur, G=3, evaluator=evaluator)
    C, L = 7, K + 10
    tidx = np.array([2, 0, 1, 1, 0, 2, 0])
    th0 = S.theta0(C, 23)
    dev = torch.device("cuda", 0)
    ch = S.chain(C)
    ch.set_statistics(2, 2, 0)
    ch.set_target_index(tidx)

    def run():
        t0 = torch.from_numpy(th0).to(dev)
        logs = []
        for part, first in ((10, True), (14, False)):
            tl = torch.zeros((part, C, L), dtype=torch.float64, device=dev)
            ch.run_device(C, part, t0.data_ptr() if first else None, seed=23, log_theta=tl.data_ptr())
            logs.append(tl.cpu().numpy())
        maps = [ch.statistics(c) for c in list(range(C)) + [-1]]
        return np.concatenate(logs), maps

    ch.schedule("eager")
    want, want_maps = run()
    ch.schedule("lazy")
    got, got_maps = run()
    lazy, cnt = ch.schedule()
    assert lazy and cnt[2] > 0
    assert np.array_equal(got, want)
    for a, b in zip(got_maps, want_maps):
        for k in ("mean", "cov", "total_variance", "normal_variance", "n"):
            assert np.array_equal(a[k], b[k], equal_nan=True), k
    # and the plain run of the same handle
    want, got, lazy, _ = _both(ch, lambda: ch.run(th0, 16, seed=29, target_index=tidx))
    assert lazy
    _assert_equal(want, got, "3 targets")
    ch.close(); S.close()


def test_certified_and_fallback_steps(ctx, femur):
    """A random walk wide enough that its density no longer dominates every step: one run takes both branches (certified and
    fallback factorisations), and its log still equals the eager schedule's."""
    C, n = 64, 24
    for sd in (0.5, 0.4, 0.6, 0.3, 0.8):
        S = Setup(ctx, femur, sd=sd)
        th0 = S.theta0(C, 11)
        ch = S.chain(C)
        want, got, lazy, cnt = _both(ch, lambda: ch.run(th0, n, seed=11))
        assert lazy
        _assert_equal(want, got, f"sd = {sd}")
        ch.close(); S.close()
        if cnt[1] > 0 and cnt[2] > 0:
            assert cnt[1] + cnt[2] == C * n
            return
    pytest.fail("no random-walk std-dev took both branches")


def test_icp_only_mixture_keeps_eager_schedule(ctx, femur):
    S = Setup(ctx, femur, icp_only=True)
    C = 16
    th0 = S.theta0(C, 3)
    ch = S.chain(C)
    want, got, lazy, cnt = _both(ch, lambda: ch.run(th0, 10, seed=3))
    assert not lazy and cnt == [0, 0, 0]
    _assert_equal(want, got, "ICP-only")
    ch.close(); S.close()


def test_lookahead_keeps_eager_schedule(ctx, femur):
    S = Setup(ctx, femur)
    C = 8
    th0 = S.theta0(C, 3)
    ch = S.chain(C)
    ch.set_lookahead(4)
    out = ch.run(th0, 10, seed=3)
    lazy, _ = ch.schedule()
    assert not lazy and out["n_accepted"].sum() > 0
    ch.close(); S.close()


def test_non_finite_observations(ctx, femur):
    """Chains whose states give non-finite observations are never certified: logs and status words equal the eager
    schedule's."""
    S = Setup(ctx, femur)
    C = 12
    th0 = S.theta0(C, 9)
    th0[3, 10:] = 1e300
    th0[7, 10] = np.inf
    ch = S.chain(C)
    want, got, lazy, cnt = _both(ch, lambda: ch.run(th0, 10, seed=9, raise_on_status=False))
    assert lazy
    _assert_equal(want, got, "non-finite observations")
    assert want["status_code"] == got["status_code"]
    ch.close(); S.close()
