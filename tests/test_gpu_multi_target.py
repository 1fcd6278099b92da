"""Chain handles over several targets (icp_chain_create_targets / icp_chain_set_target_index): every chain of a multi-target
run equals the single-target run of that chain on its own target, bit for bit, on the runner's paths (step by step,
rejection look-ahead, resumed runs, statistics) and rank updates; the oracle per chain; targets of different vertex counts
and with a boundary; the argument checks."""
import numpy as np
import pytest

from icp_proposal_b200 import _lib, core, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

K = 101
KEYS = ("component", "accepted", "values", "theta", "theta_final", "n_accepted", "status", "theta_best", "value_best")


def _base(femur):
    return dict(ref=femur["ref"], cells=femur["cells"], **femur["gpmm_100"])


def _perturbed(base, t_index):
    """The perturbed femur-twin targets of test_config4_hausdorff_chains_on_perturbed_targets."""
    target = synth.model_instance(base, np.random.default_rng(100 + t_index).normal(0, 1.0, K))
    return target + np.random.default_rng(7 + t_index).normal(0, 0.5, target.shape), base["cells"]


def _split_centroids(verts, cells, k):
    """A closed mesh with k more vertices: the first k triangles split at their centroids."""
    v, c = [verts], [cells[k:]]
    for i in range(k):
        a, b, d = cells[i]
        n = len(verts) + i
        v.append(verts[cells[i]].mean(0, keepdims=True))
        c.append(np.array([[a, b, n], [b, d, n], [d, a, n]], np.int32))
    return np.concatenate(v), np.concatenate(c).astype(np.int32)


class Set:
    """Model + G targets, each with the config-1 mixture and an evaluator; entry g as core.Chain's targets list."""

    def __init__(self, ctx, base, meshes, evaluator="hausdorff", rank_update=_lib.RANK_UPDATE_FP64, n_eval=4 * K):
        self.model = core.Model(ctx, base["ref"], base["cells"], base["basis"], base["variance"])
        self.meshes, self.entries, self.handles = meshes, [], []
        ids, eids = np.arange(2 * K), np.arange(n_eval)
        for tv, tc in meshes:
            tgt = core.Target(ctx, tv, tc)
            tp = tv[:: len(tv) // (2 * K)][: 2 * K]
            mk = lambda d: core.IcpProposal(self.model, tgt, 0.1, 10.0, 5.0, d, True, ids, tp, rank_update=rank_update)
            pt, pm = mk(_lib.TARGET_SAMPLING), mk(_lib.MODEL_SAMPLING)
            comps = [dict(kind=0, weight=0.45, proposal=pt), dict(kind=0, weight=0.45, proposal=pm), dict(kind=1, weight=0.1, sd=0.1)]
            if evaluator == "hausdorff":
                ev = core.Evaluator(self.model, tgt, _lib.EVAL_HAUSDORFF, 0, True, 100.0)
            elif evaluator == "independent":
                ev = core.Evaluator(self.model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 2.0, 0.0, eids, tp)
            else:
                ev = core.Evaluator(self.model, tgt, _lib.EVAL_COLLECTIVE, _lib.SYMMETRIC, True, 0.1, 2.0, 1.0, eids, tp)
            self.entries.append((tgt, comps, ev))
            self.handles += [ev, pt, pm, tgt]

    def chain(self, C, width, which=None):
        ents = self.entries if which is None else [self.entries[which]]
        ch = core.Chain(self.model, targets=ents, max_chains=C) if len(ents) > 1 else core.Chain(self.model, *ents[0], C)
        ch.set_lookahead(width)
        return ch

    def theta0(self, C, seed):
        rng = np.random.default_rng(seed)
        return np.stack([self.model.theta()] + [self.model.theta(rng.normal(0, np.sqrt(0.1), K)) for _ in range(C - 1)])

    def close(self):
        for h in self.handles:
            h.close()
        self.model.close()


def _assert_chain_equal(multi, single, c, what):
    for k in KEYS:
        a, b = multi[k], single[k]
        a = a[:, c] if k in ("component", "accepted", "values", "theta") else a[c]
        b = b[:, 0] if k in ("component", "accepted", "values", "theta") else b[0]
        assert np.array_equal(a, b, equal_nan=True), f"{k} of chain {c} differs ({what})"


def _check_batch_independence(S, C, n, width, seed=31, tidx=None):
    tidx = np.arange(C) % len(S.entries) if tidx is None else tidx
    th0 = S.theta0(C, seed)
    ch = S.chain(C, width)
    multi = ch.run(th0, n, seed=seed, target_index=tidx)
    ch.close()
    assert 0 < multi["n_accepted"].sum() < C * n
    singles = [S.chain(1, width, which=g) for g in range(len(S.entries))]
    for c in range(C):
        single = singles[tidx[c]].run(th0[c:c + 1], n, seed=seed, chain_id_offset=c)
        _assert_chain_equal(multi, single, c, f"width {width}")
    for s in singles:
        s.close()
    return multi


@pytest.mark.parametrize("evaluator", ["independent", "hausdorff"])
@pytest.mark.parametrize("width", [0, 4])
@pytest.mark.parametrize("rank_update", [_lib.RANK_UPDATE_FP64, _lib.RANK_UPDATE_INT8])
def test_chains_equal_their_single_target_runs(ctx, femur, evaluator, width, rank_update):
    """G = 3 perturbed femur targets, interleaved target indices: every chain's log, final state, counters, status and best
    sample equal those of its single-target run with the same seed and global chain id."""
    base = _base(femur)
    S = Set(ctx, base, [_perturbed(base, t) for t in range(3)], evaluator, rank_update)
    _check_batch_independence(S, 6, 24, width)
    S.close()


def test_int8_single_target_runs_are_batch_invariant(ctx, femur):
    """The premise of the INT8 case above on one target: chain c of a batch equals the same chain run alone at
    chain_id_offset c."""
    base = _base(femur)
    S = Set(ctx, base, [_perturbed(base, 0)], "hausdorff", _lib.RANK_UPDATE_INT8)
    C, n = 4, 20
    th0 = S.theta0(C, 5)
    ch = S.chain(C, 0)
    batch = ch.run(th0, n, seed=5)
    for c in range(C):
        _assert_chain_equal(batch, ch.run(th0[c:c + 1], n, seed=5, chain_id_offset=c), c, "INT8 single target")
    ch.close(); S.close()


def test_oracle_per_chain(ctx, femur):
    """Two targets, two chains each, caller-supplied randomness: every chain against orc.chain_run on its own target with
    the tolerances of test_config4_hausdorff_chains_on_perturbed_targets."""
    base = _base(femur)
    meshes = [_perturbed(base, t) for t in range(2)]
    S = Set(ctx, base, meshes, "hausdorff")
    C, n = 4, 15
    tidx = np.array([0, 1, 1, 0])
    rng = np.random.default_rng(21)
    th0 = S.theta0(C, 21)
    u_comp, u_acc, z = rng.random((n, C)), rng.random((n, C)), rng.normal(size=(n, C, K))
    ch = S.chain(C, 0)
    got = ch.run(th0, n, u_comp=u_comp, z=z, u_acc=u_acc, target_index=tidx)
    om = orc.Model(base["ref"], base["cells"], base["basis"], base["variance"])
    ids = np.arange(2 * K)
    for c in range(C):
        tv, tc = meshes[tidx[c]]
        ot = orc.Mesh(tv, tc)
        tp = tv[:: len(tv) // (2 * K)][: 2 * K]
        mo = lambda d: orc.IcpProposal(om, ot, 0.1, 10.0, 5.0, d, True, ids, tp)
        comps_o = [dict(kind=0, weight=0.45, icp=mo(1)), dict(kind=0, weight=0.45, icp=mo(0)), dict(kind=1, weight=0.1, sd=0.1)]
        want = orc.chain_run(om, ot, comps_o, True, orc.EVAL_HAUSDORFF, 0, (100.0,), ids, tp, th0[c], n, u_comp[:, c], z[:, c],
                             u_acc[:, c], closed_form=True)
        assert np.array_equal(got["component"][:, c], want["comp"])
        assert np.array_equal(got["accepted"][:, c], want["accepted"])
        np.testing.assert_allclose(got["values"][:, c], want["logv"], rtol=1e-7)
        np.testing.assert_allclose(got["theta"][:, c], want["theta"], rtol=0, atol=1e-7)
    ch.close(); S.close()


def test_hausdorff_targets_of_different_vertex_counts(ctx, femur):
    """Closed targets with 1622 and 1622 + 40 vertices: the shorter Hausdorff list is padded, the values are unchanged."""
    base = _base(femur)
    a = _perturbed(base, 0)
    b = _split_centroids(*_perturbed(base, 1), 40)
    S = Set(ctx, base, [a, b], "hausdorff")
    assert len(b[0]) == len(a[0]) + 40
    assert not S.entries[1][0].boundary_flags().any()
    for width in (0, 4):
        _check_batch_independence(S, 4, 20, width, seed=41)
    S.close()


def test_open_target_with_the_collective_evaluator(ctx, femur):
    """A closed target and a partial (open) one of the same model: the set takes the boundary path for both, so the closed
    target's chains agree with their single-target runs to rounding; the open target's chains are bit-identical."""
    base = _base(femur)
    tv, tc, _ = synth.partial_target(base, seed=5, alpha_sd=0.3)
    meshes = [_perturbed(base, 0), (tv, tc)]
    S = Set(ctx, base, meshes, "collective", n_eval=2 * K)
    assert S.entries[1][0].boundary_flags().any() and not S.entries[0][0].boundary_flags().any()
    C, n, seed = 4, 20, 51
    tidx = np.array([0, 1, 0, 1])
    th0 = S.theta0(C, seed)
    ch = S.chain(C, 0)
    multi = ch.run(th0, n, seed=seed, target_index=tidx)
    assert 0 < multi["n_accepted"].sum() < C * n
    for c in range(C):
        one = S.chain(1, 0, which=tidx[c])
        single = one.run(th0[c:c + 1], n, seed=seed, chain_id_offset=c)
        one.close()
        if tidx[c] == 1:
            _assert_chain_equal(multi, single, c, "open target")
        else:
            assert np.array_equal(multi["accepted"][:, c], single["accepted"][:, 0])
            np.testing.assert_allclose(multi["values"][:, c], single["values"][:, 0], rtol=1e-12, atol=0)
    ch.close(); S.close()


def test_resume_and_statistics_on_a_target_set(ctx, femur):
    """A run split 12 + 18 through the resumed device runner, with statistics on, equals the uninterrupted run: the log and
    every chain's maps bit for bit."""
    import torch
    base = _base(femur)
    S = Set(ctx, base, [_perturbed(base, t) for t in range(3)], "hausdorff")
    C, n, L = 5, 30, K + 10
    tidx = np.array([2, 0, 1, 1, 0])
    th0 = S.theta0(C, 61)
    stats = (3, 2, 0)
    full = S.chain(C, 0)
    full.set_statistics(*stats)
    want = full.run(th0, n, seed=61, target_index=tidx)
    want_maps = [full.statistics(c) for c in list(range(C)) + [-1]]
    dev = torch.device("cuda", 0)
    for width in (0, 4):
        ch = S.chain(C, width)
        ch.set_statistics(*stats)
        ch.set_target_index(tidx)
        t0 = torch.from_numpy(th0).to(dev)
        logs = []
        for part, first in ((12, True), (18, False)):
            tl = torch.zeros((part, C, L), dtype=torch.float64, device=dev)
            ch.run_device(C, part, t0.data_ptr() if first else None, seed=61, log_theta=tl.data_ptr())
            logs.append(tl.cpu().numpy())
        assert np.array_equal(np.concatenate(logs), want["theta"]), f"width {width}"
        for a, b in zip([ch.statistics(c) for c in list(range(C)) + [-1]], want_maps):
            for k in ("mean", "cov", "total_variance", "normal_variance", "n"):
                assert np.array_equal(a[k], b[k], equal_nan=True), f"{k} differs (width {width})"
        ch.close()
    full.close(); S.close()


def test_argument_checks_and_references(ctx, femur):
    base = _base(femur)
    S = Set(ctx, base, [_perturbed(base, t) for t in range(2)], "hausdorff")
    model, (t0, c0, e0), (t1, c1, e1) = S.model, S.entries[0], S.entries[1]

    def refused(entries, field):
        with pytest.raises(_lib.IcpCudaError) as ex:
            core.Chain(model, targets=entries, max_chains=4)
        assert ex.value.code == _lib.ERR_INVALID_ARGUMENT and field in str(ex.value), str(ex.value)

    ids = np.arange(2 * K)
    refused([(t0, c0, e0), (t1, [dict(c1[0], weight=0.5)] + c1[1:], e1)], "component 0 weight")
    refused([(t0, c0, e0), (t1, c1[:2] + [dict(c1[2], sd=0.2)], e1)], "component 2 sd")
    refused([(t0, c0, e0), (t1, c1[:2] + [dict(kind=3, weight=0.1, sd=0.1)], e1)], "component 2 kind")
    tv1 = S.meshes[1][0]
    tp1 = tv1[:: len(tv1) // (2 * K)][: 2 * K]
    others = []
    for kw, field in ((dict(step_length=0.2), "step_length"), (dict(ids=ids[::-1].copy()), "model point ids"),
                      (dict(tp=tp1[:-1]), "n_tp"), (dict(boundary_aware=False), "boundary_aware")):
        a = dict(step_length=0.1, boundary_aware=True, ids=ids, tp=tp1)
        a.update(kw)
        p = core.IcpProposal(model, t1, a["step_length"], 10.0, 5.0, _lib.TARGET_SAMPLING, a["boundary_aware"], a["ids"], a["tp"])
        others.append(p)
        refused([(t0, c0, e0), (t1, [dict(c1[0], proposal=p)] + c1[1:], e1)], "proposal " + field)
    ev_rate = core.Evaluator(model, t1, _lib.EVAL_HAUSDORFF, 0, True, 50.0)
    ev_kind = core.Evaluator(model, t1, _lib.EVAL_INDEPENDENT, 0, True, 0.0, 2.0, 0.0, ids, tp1)
    refused([(t0, c0, e0), (t1, c1, ev_rate)], "evaluator p0")
    refused([(t0, c0, e0), (t1, c1, ev_kind)], "evaluator kind")
    refused([(t0, c0, e0), (t1, c1, e0)], "evaluator was built for another")   # e0 belongs to target 0
    ch = core.Chain(model, targets=[(t0, c0, e0), (t1, c1, e1)], max_chains=4)
    th0 = S.theta0(3, 1)
    with pytest.raises(_lib.IcpCudaError, match="set_target_index"):
        ch.run(th0, 2)                                                         # no target index yet
    for bad in ([0, 1], [0, 2, 1], [0, -1, 1], [0] * 5):
        with pytest.raises(_lib.IcpCudaError):
            ch.set_target_index(bad) if len(bad) != 2 else ch.run(th0, 2, target_index=bad)
    with pytest.raises(_lib.IcpCudaError, match="metrics_interval"):
        ch.run(th0, 4, target_index=[0, 1, 0], metrics_interval=2)
    ch.run(th0, 2, target_index=[0, 1, 0])
    # the handle holds references on every entry's target, proposals and evaluator; destroying the chain releases them
    lib = model.lib
    assert lib.icp_target_destroy(t1.h) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_evaluator_destroy(e1.h) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_proposal_destroy(c1[1]["proposal"].h) == _lib.ERR_INVALID_ARGUMENT
    ch.close()
    for h in others + [ev_rate, ev_kind]:
        h.close()
    for h in S.handles:
        destroy = {core.Evaluator: lib.icp_evaluator_destroy, core.IcpProposal: lib.icp_proposal_destroy,
                   core.Target: lib.icp_target_destroy}[type(h)]
        assert destroy(h.h) == _lib.OK
        h.h = None
    assert lib.icp_model_destroy(model.h) == _lib.OK
    model.h = None
