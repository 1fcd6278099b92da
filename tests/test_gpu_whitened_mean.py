"""The chain runner keeps y = L^-1 b in a posterior's mean slot instead of mu = L^-T y, so its factorisations skip the back
substitution. Checked here: both forms of every factorisation path on the same matrices (L bit-identical, y = L^T mu, the
same backward transition form), and chains whose proposals and accept decisions match the per-call entry points, which
keep mu."""
import numpy as np
import pytest

from conftest import random_theta
from icp_proposal_b200 import _lib, core

pytestmark = pytest.mark.gpu

STEP = 0.1


def _dev(ctx, m):
    return core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])


def _femur(femur, which):
    return dict(ref=femur["ref"], cells=femur["cells"], target=femur["target"], target_cells=femur["target_cells"], **femur[which])


@pytest.mark.parametrize("which,rank_update", [("gpmm_100", _lib.RANK_UPDATE_INT8), ("gpmm_100", _lib.RANK_UPDATE_FP64),
                                               ("gpmm_200", _lib.RANK_UPDATE_FP64)])
def test_factor_forms_agree(ctx, femur, which, rank_update):
    """K = 101 runs k_cholesky_packed, K = 201 the large-rank pair (k_pack_lower + k_cholesky_packed)."""
    m = _femur(femur, which)
    K = len(m["variance"])
    model, tgt = _dev(ctx, m)
    rng = np.random.default_rng(5)
    C = 4
    th = random_theta(m, rng, C)
    ids = np.arange(2 * K)
    tp = m["target"][:: len(m["target"]) // (2 * K)][: 2 * K]
    prop = core.IcpProposal(model, tgt, STEP, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=rank_update)
    mu, M, _ = prop.posterior(th)
    b = np.einsum("cij,cj->ci", M, mu)
    to = prop.propose(th, rng.normal(size=(C, K)))
    L0, mu0, q0, st0 = ctx.factor(M, b, th, to, STEP, ymean=False)
    L1, y1, q1, st1 = ctx.factor(M, b, th, to, STEP, ymean=True)
    assert np.all(st0 == 0) and np.all(st1 == 0)
    assert np.array_equal(L0, L1)
    Lty = np.einsum("cij,ci->cj", L0, mu0)
    assert np.abs(y1 - Lty).max() <= 1e-12 * np.abs(y1).max()
    np.testing.assert_allclose(q1, q0, rtol=1e-11)
    # the per-call transition density (its own posterior of th, mu form)
    lt = prop.log_transition(th, to)
    np.testing.assert_allclose(q1, -2.0 * lt - K * np.log(2 * np.pi), rtol=1e-9)
    # without transition arguments the mean slot is the same
    _, y2, q2, _ = ctx.factor(M, b, ymean=True)
    assert q2 is None and np.array_equal(y1, y2)
    prop.close(); model.close(); tgt.close()


@pytest.mark.parametrize("K", [61, 131])
def test_factor_forms_agree_synthetic(ctx, K):
    """Random posterior-like matrices I + AᵀA: K = 131 runs k_cholesky_solve_mma (104 < Kp <= 160)."""
    rng = np.random.default_rng(K)
    C = 3
    A = rng.normal(size=(C, 2 * K, K))
    M = np.eye(K) + np.einsum("cri,crj->cij", A, A)
    b = rng.normal(size=(C, K)) * 10.0
    th = np.zeros((C, K + 10)); th[:, 10:] = rng.normal(size=(C, K))
    to = th.copy(); to[:, 10:] += 0.1 * rng.normal(size=(C, K))
    L0, mu0, q0, st0 = ctx.factor(M, b, th, to, STEP, ymean=False)
    L1, y1, q1, st1 = ctx.factor(M, b, th, to, STEP, ymean=True)
    assert np.all(st0 == 0) and np.all(st1 == 0)
    assert np.array_equal(L0, L1)
    np.testing.assert_allclose(mu0, np.linalg.solve(M, b[..., None])[..., 0], rtol=1e-9, atol=1e-12 * np.abs(mu0).max())
    assert np.abs(y1 - np.einsum("cij,ci->cj", L0, mu0)).max() <= 1e-12 * np.abs(y1).max()
    np.testing.assert_allclose(q1, q0, rtol=1e-11)


def _lse(ls, w):
    ls = np.asarray(ls); mx = ls.max()
    return -np.inf if not np.isfinite(mx) else mx + np.log(np.sum(w * np.exp(ls - mx)))


@pytest.mark.parametrize("mixture", ["icp_rw", "icp_only", "svd"])
def test_chain_matches_per_call_entry_points(ctx, twin31, mixture):
    """Every step of a chain with caller-supplied randomness: the proposal (logged when accepted) against icp_propose, and
    the accept decision against one formed from icp_log_transition. "svd": one component samples through the reference's
    SVD factor, whose mean slot keeps mu, next to a Cholesky component."""
    m = twin31
    K = len(m["variance"])
    model, tgt = _dev(ctx, m)
    ids, eids = np.arange(2 * K), np.arange(4 * K)
    tp = m["target"][:: len(m["target"]) // (2 * K)][: 2 * K]
    f0 = _lib.FACTOR_SVD if mixture == "svd" else _lib.FACTOR_CHOLESKY
    p0 = core.IcpProposal(model, tgt, STEP, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp, factor=f0)
    p1 = core.IcpProposal(model, tgt, STEP, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp)
    w = np.array([0.45, 0.45, 0.1]) if mixture == "icp_rw" else np.array([0.5, 0.5])
    sd = 0.1
    comps = [dict(kind=_lib.PROP_ICP, weight=w[0], proposal=p0), dict(kind=_lib.PROP_ICP, weight=w[1], proposal=p1)]
    if len(w) == 3:
        comps.append(dict(kind=_lib.PROP_RANDOM_SHAPE, weight=w[2], sd=sd))
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
    chain = core.Chain(model, tgt, comps, ev, max_chains=1)
    rng = np.random.default_rng(11)
    n = 40
    th0 = model.theta(rng.normal(0, 0.5, K))[None]
    u_comp, u_acc, z = rng.random((n, 1)), rng.random((n, 1)), rng.normal(size=(n, 1, K))
    got = chain.run(th0, n, u_comp=u_comp, z=z, u_acc=u_acc)
    cur, vcur = th0.copy(), ev.log_value(th0)[0, 0]
    n_icp_acc = 0
    for s in range(n):
        ci = int(got["component"][s, 0])
        if ci < 2:
            prop = (p0, p1)[ci].propose(cur, z[s])
        else:
            prop = cur.copy(); prop[0, 10:] += sd * z[s, 0]
        vprop = ev.log_value(prop)[0, 0]
        fwd = [p0.log_transition(cur, prop)[0], p1.log_transition(cur, prop)[0]]
        bwd = [p0.log_transition(prop, cur)[0], p1.log_transition(prop, cur)[0]]
        if len(w) == 3:
            d2 = float(np.sum((prop[0, 10:] - cur[0, 10:]) ** 2))
            rw = -0.5 * (K * np.log(2 * np.pi) + K * np.log(sd * sd) + d2 / (sd * sd))
            fwd.append(rw); bwd.append(rw)
        a = vprop - vcur - (_lse(fwd, w) - _lse(bwd, w))
        assert ((a > 0) or (u_acc[s, 0] < np.exp(a))) == bool(got["accepted"][s, 0]), s
        if got["accepted"][s, 0]:
            np.testing.assert_allclose(got["theta"][s, 0], prop[0], rtol=1e-10, atol=1e-10 * np.abs(prop[0]).max())
            n_icp_acc += ci < 2
            cur, vcur = got["theta"][s:s + 1, 0].copy(), got["values"][s, 0, 0]
    assert n_icp_acc > 0
    chain.close(); ev.close(); p0.close(); p1.close(); model.close(); tgt.close()
