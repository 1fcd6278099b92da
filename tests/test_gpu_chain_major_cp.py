"""Chain-major closest-point queries (k_nearest takes the same query row of consecutive chains in consecutive lanes): a batch of
C chains equals C one-chain calls bit for bit - evaluator values on the static model -> target and the dynamic target -> model
paths, model-sampling proposals, seeded second calls, a NaN state, and chains of three interleaved targets."""
import numpy as np
import pytest

from icp_proposal_b200 import _lib, core, synth

pytestmark = pytest.mark.gpu

K = 101
CHAINS = (1, 5, 31, 32, 33, 257)


def _target(base, t_index=0):
    target = synth.model_instance(base, np.random.default_rng(100 + t_index).normal(0, 1.0, K))
    return target + np.random.default_rng(7 + t_index).normal(0, 0.5, target.shape), base["cells"]


@pytest.fixture(scope="module")
def setup(ctx, femur):
    base = dict(ref=femur["ref"], cells=femur["cells"], **femur["gpmm_100"])
    model = core.Model(ctx, base["ref"], base["cells"], base["basis"], base["variance"])
    tv, tc = _target(base)
    tgt = core.Target(ctx, tv, tc)
    yield base, model, tgt, tv
    tgt.close()
    model.close()


def _thetas(model, C, seed, sd=0.3):
    rng = np.random.default_rng(seed)
    return np.stack([model.theta(rng.normal(0, sd, K), translation=rng.normal(0, 2.0, 3)) for _ in range(C)])


def _per_chain(f, th):
    return np.concatenate([f(th[c:c + 1]) for c in range(len(th))])


@pytest.mark.parametrize("C", CHAINS)
@pytest.mark.parametrize("mode", [_lib.MODEL_TO_TARGET, _lib.TARGET_TO_MODEL])
@pytest.mark.parametrize("n_eval", [404, 77])
def test_evaluator_batch_equals_single_chain_calls(setup, C, mode, n_eval):
    """Independent evaluator, model -> target (static target BVH, Morton-permuted query rows) and target -> model (refitted
    per-chain model BVHs, every lane of a warp on the same target point); 77 query rows are not a multiple of 32. The second
    call starts from the seeds the first one left, the third carries a NaN state in its middle chain."""
    base, model, tgt, tv = setup
    eids = np.linspace(0, len(base["ref"]) - 1, n_eval).astype(np.int32)
    tp = tv[:: len(tv) // n_eval][:n_eval]
    batch = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, mode, True, 0.0, 2.0, 0.0, eids, tp)
    single = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, mode, True, 0.0, 2.0, 0.0, eids, tp)
    th = _thetas(model, C, 11 + C)
    th2 = th + np.random.default_rng(C).normal(0, 0.05, th.shape) * (np.arange(th.shape[1]) >= 10)
    th3 = th2.copy()
    th3[C // 2, 12] = np.nan
    for k, t in enumerate((th, th2, th3)):
        got = batch.log_value(t)
        want = _per_chain(single.log_value, t)
        assert np.array_equal(got, want, equal_nan=True), f"call {k}, C = {C}"
        if k < 2:
            assert np.isfinite(got).all()
        else:
            assert np.isnan(got[C // 2, 2]) and np.isfinite(np.delete(got, C // 2, axis=0)).all()
    batch.close()
    single.close()


@pytest.mark.parametrize("C", CHAINS)
def test_model_sampling_proposal_batch_equals_single_chain_calls(setup, C):
    """Model-sampling ICP proposal (closest target points of 202 model points per chain, seeded from the previous call):
    posterior means and proposals of a batch equal the one-chain calls, on two successive calls."""
    base, model, tgt, tv = setup
    ids = np.linspace(0, len(base["ref"]) - 1, 2 * K).astype(np.int32)   # 202 points spread over the whole mesh
    tp = tv[:: len(tv) // (2 * K)][: 2 * K]
    mk = lambda: core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp)
    batch, single = mk(), mk()
    rng = np.random.default_rng(3 + C)
    th = _thetas(model, C, 5 + C)
    for k in range(2):
        z = rng.normal(size=(C, K))
        mu, _, n = batch.posterior(th, want_M=False)
        for c in range(C):
            mu1, _, n1 = single.posterior(th[c:c + 1], want_M=False)
            assert np.array_equal(mu[c], mu1[0]) and n[c] == n1[0], f"posterior of chain {c}, call {k}, C = {C}"
        got = batch.propose(th, z)
        want = np.concatenate([single.propose(th[c:c + 1], z[c:c + 1]) for c in range(C)])
        assert np.array_equal(got, want), f"call {k}, C = {C}"
        th = got
    batch.close()
    single.close()


def test_three_interleaved_targets(ctx, setup):
    """33 chains over three targets, target index c % 3, so the lanes of every warp of the model -> target queries walk three
    different trees: every chain's log equals its single-target run."""
    base, model, _, _ = setup
    ids, eids = np.arange(2 * K), np.arange(4 * K)
    handles, entries = [], []
    for t in range(3):
        tv, tc = _target(base, t)
        tgt = core.Target(ctx, tv, tc)
        tp = tv[:: len(tv) // (2 * K)][: 2 * K]
        mk = lambda d: core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, d, True, ids, tp)
        pt, pm = mk(_lib.TARGET_SAMPLING), mk(_lib.MODEL_SAMPLING)
        comps = [dict(kind=0, weight=0.45, proposal=pt), dict(kind=0, weight=0.45, proposal=pm), dict(kind=1, weight=0.1, sd=0.1)]
        ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
        entries.append((tgt, comps, ev))
        handles += [ev, pt, pm, tgt]
    C, n, seed = 33, 12, 17
    tidx = np.arange(C) % 3
    rng = np.random.default_rng(seed)
    th0 = np.stack([model.theta(rng.normal(0, np.sqrt(0.1), K)) for _ in range(C)])
    multi_ch = core.Chain(model, targets=entries, max_chains=C)
    multi = multi_ch.run(th0, n, seed=seed, target_index=tidx)
    multi_ch.close()
    assert 0 < multi["n_accepted"].sum() < C * n
    singles = [core.Chain(model, *entries[g], 1) for g in range(3)]
    for c in range(C):
        one = singles[tidx[c]].run(th0[c:c + 1], n, seed=seed, chain_id_offset=c)
        for k in ("component", "accepted", "values", "theta"):
            assert np.array_equal(multi[k][:, c], one[k][:, 0], equal_nan=True), f"{k} of chain {c}"
        for k in ("theta_final", "n_accepted"):
            assert np.array_equal(multi[k][c], one[k][0], equal_nan=True), f"{k} of chain {c}"
    for s in singles:
        s.close()
    for h in handles:
        h.close()
