"""Posterior variability maps accumulated inside the fused chain runner (icp_chain_set_statistics / icp_chain_statistics)
against icp_posterior_variability over the selected rows of the chain log, the bit identity of the maps across the runner's
paths (step by step, rejection look-ahead, resumed runs), the unchanged chain log, sharding and the argument checks."""
import numpy as np
import pytest

from conftest import random_theta
from icp_proposal_b200 import _lib, api, core, sharding, synth
from oracle import np_oracle as npo

pytestmark = pytest.mark.gpu

KEYS = ("mean", "cov", "total_variance", "normal_variance")


def _selected(n_steps, burn_in, every, end):
    return np.arange(burn_in, min(n_steps, end) if end > 0 else n_steps, every)


def _assert_maps(got, want, rtol=1e-9):
    for k in KEYS:
        w = np.asarray(want[k])
        # entries that cancel to ~0 (off-diagonal covariances) are compared on the scale of the map
        np.testing.assert_allclose(got[k], w, rtol=rtol, atol=rtol * np.abs(w).max(), err_msg=k)


def _assert_equal(a, b, what):
    for k in KEYS + ("n",):
        assert np.array_equal(a[k], b[k], equal_nan=True), f"{k} differs ({what})"


@pytest.fixture(scope="module")
def mix(ctx, twin31):
    """ICP in both directions, random walk and pose components (the mixture of test_rejection_lookahead_is_bit_identical)."""
    m = twin31
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, m["target"], m["target_cells"])
    ids, tp = np.arange(62), m["target"][::26][:62]
    pt = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.TARGET_SAMPLING, True, ids, tp)
    pm = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, rank_update=_lib.RANK_UPDATE_INT8)
    comps = [dict(kind=_lib.PROP_ICP, weight=0.3, proposal=pt), dict(kind=_lib.PROP_ICP, weight=0.3, proposal=pm),
             dict(kind=_lib.PROP_RANDOM_SHAPE, weight=0.3, sd=0.15), dict(kind=2, weight=0.05, sd=0.01, axis=1),
             dict(kind=3, weight=0.05, sd=0.2, axis=0)]
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, _lib.MODEL_TO_TARGET, True, 0.0, 1.0, 0.0, np.arange(124), tp)
    yield m, model, tgt, comps, ev
    ev.close(); pt.close(); pm.close(); model.close(); tgt.close()


def _chain(mix, C, width=-1, stats=None):
    m, model, tgt, comps, ev = mix
    ch = core.Chain(model, tgt, comps, ev, max_chains=C)
    ch.set_lookahead(width)
    if stats is not None:
        ch.set_statistics(*stats)
    return ch


@pytest.mark.parametrize("burn_in,every,end", [(0, 1, 0), (7, 3, 40), (25, 5, 0), (3, 10, 55)])
def test_maps_match_the_chain_log(mix, burn_in, every, end):
    """Per-chain and pooled maps equal icp_posterior_variability over log_theta[selected] (the state current after each
    selected step), with the direction of normal_variance from the samples' normals or from a reference state."""
    m, model = mix[0], mix[1]
    C, n = 4, 60
    th0 = random_theta(m, np.random.default_rng(11), C, alpha_sd=0.4, pose=True)
    ch = _chain(mix, C, stats=(burn_in, every, end))
    run = ch.run(th0, n, seed=5)
    sel = _selected(n, burn_in, every, end)
    rate = run["n_accepted"].mean() / n
    assert 0.05 < rate < 0.95
    if burn_in == 25:   # the burn-in lies past the first acceptance of some chain, so its first sample is not theta0
        assert run["accepted"][:burn_in].any(axis=0).any()
    assert np.ptp(run["theta"][:, :, 1:7], axis=0).max() > 0      # the pose varies
    for sum_normals, ref in ((True, None), (False, None), (False, th0[1])):
        for c in list(range(C)) + [-1]:
            got = ch.statistics(c, sum_normals, ref)
            thetas = run["theta"][sel, c] if c >= 0 else run["theta"][sel].reshape(-1, model.K + 10)
            assert got["n"] == len(thetas)
            _assert_maps(got, core.posterior_variability(model, thetas, sum_normals, ref))
    # reading leaves the accumulators unchanged
    _assert_equal(ch.statistics(-1), ch.statistics(-1), "second read")
    ch.close()


def test_maps_match_the_oracle(mix):
    """One case against the loop-for-loop restatement of PosteriorVariability.scala on the reconstructed meshes."""
    m, model = mix[0], mix[1]
    C, n = 2, 40
    th0 = random_theta(m, np.random.default_rng(12), C, alpha_sd=0.4, pose=True)
    ch = _chain(mix, C, stats=(4, 2, 0))
    run = ch.run(th0, n, seed=8)
    sel = _selected(n, 4, 2, 0)
    for sum_normals in (True, False):
        got = ch.statistics(1, sum_normals, None if sum_normals else th0[0])
        meshes = list(model.reconstruct(run["theta"][sel, 1]))
        want = npo.posterior_variability(meshes, m["cells"], ref_verts=model.reconstruct(th0[0])[0], sum_normals=sum_normals)
        _assert_maps(got, dict(zip(KEYS, want)))
    ch.close()


def test_reference_selection_walks_back_to_accepted_records(mix):
    """LogHelper.samplesFromLog picks, for every selected index, the last accepted record at or before it: with an accepted
    record before the first selected index, icp_chainlog_sample_indices + log_theta gives the same maps."""
    m, model = mix[0], mix[1]
    C, n, burn_in, every, end = 4, 50, 12, 4, 45
    th0 = random_theta(m, np.random.default_rng(13), C, alpha_sd=0.4)
    ch = _chain(mix, C, stats=(burn_in, every, end))
    run = ch.run(th0, n, seed=9)
    checked = walked = 0
    for c in range(C):
        st = run["accepted"][:, c]
        if not st[:burn_in].any():
            continue
        idx = core.chainlog_sample_indices(st, take_every_n=every, total=end, burn_in=burn_in)
        walked += int((idx != _selected(n, burn_in, every, end)).any())
        for sum_normals in (True, False):
            _assert_maps(ch.statistics(c, sum_normals), core.posterior_variability(model, run["theta"][idx, c], sum_normals))
        checked += 1
    assert checked >= 1 and walked >= 1
    ch.close()


def test_maps_are_bit_identical_across_runner_paths(mix):
    """The step-by-step runner, the look-ahead at widths 2, 8 and automatic, and a run split 20 + 25 through the resumed
    device runner present the same (state, weight) updates: the maps are equal, not merely close."""
    import torch
    m = mix[0]
    C, n, L = 3, 45, 41
    th0 = random_theta(m, np.random.default_rng(14), C, alpha_sd=0.4, pose=True)
    stats = (2, 3, 0)

    def read(ch):
        return [ch.statistics(c, sn) for c in list(range(C)) + [-1] for sn in (True, False)]

    ref_ch = _chain(mix, C, 0, stats)
    run = ref_ch.run(th0, n, seed=77)
    assert ref_ch.last_run_rounds() == n and 0 < run["n_accepted"].sum() < C * n
    want = read(ref_ch)
    ref_ch.close()
    for width in (2, 8, -1):
        ch = _chain(mix, C, width, stats)
        got = ch.run(th0, n, seed=77)
        assert np.array_equal(got["theta"], run["theta"])
        if width > 0:
            assert ch.last_run_rounds() < n
        for a, b in zip(read(ch), want):
            _assert_equal(a, b, f"width {width}")
        ch.close()
    dev = torch.device("cuda", 0)
    for width in (0, -1):
        ch = _chain(mix, C, width, stats)
        t0 = torch.from_numpy(th0).to(dev)
        for part, first in ((20, True), (25, False)):
            tl = torch.zeros((part, C, L), dtype=torch.float64, device=dev)
            ch.run_device(C, part, t0.data_ptr() if first else None, seed=77, log_theta=tl.data_ptr())
        for a, b in zip(read(ch), want):
            _assert_equal(a, b, f"resumed run, width {width}")
        ch.close()


@pytest.mark.parametrize("width", [0, 4])
def test_chain_log_is_unchanged_by_statistics(mix, width):
    """Every output of test_rejection_lookahead_is_bit_identical is bit-identical with statistics on and off."""
    m = mix[0]
    C, n, K = 3, 45, 31
    rng = np.random.default_rng(15)
    th0 = random_theta(m, rng, C, alpha_sd=0.4)
    keys = ("component", "accepted", "values", "theta", "theta_final", "n_accepted", "theta_best", "value_best", "status")
    for kw in (dict(seed=77), dict(u_comp=rng.random((n, C)), z=rng.normal(size=(n, C, K)), u_acc=rng.random((n, C)))):
        off = _chain(mix, C, width)
        want = off.run(th0, n, **kw)
        on = _chain(mix, C, width, (0, 1, 0))
        got = on.run(th0, n, **kw)
        for k in keys:
            assert np.array_equal(got[k], want[k], equal_nan=True), k
        assert on.statistics(-1)["n"] == C * n
        # switched off again: the next run from theta0 drops them
        on.set_statistics(None)
        again = on.run(th0, n, **kw)
        for k in keys:
            assert np.array_equal(again[k], want[k], equal_nan=True), k
        with pytest.raises(_lib.IcpCudaError):
            on.statistics(-1)
        off.close(); on.close()


def test_femur_config1_shape(ctx, femur):
    """Femur GPMM-100 with the config-1 mixture at 64 chains x 200 steps against icp_posterior_variability over the log."""
    m = dict(ref=femur["ref"], cells=femur["cells"], target=femur["target"], target_cells=femur["target_cells"], **femur["gpmm_100"])
    K = 101
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, m["target"], m["target_cells"])
    ids, eids = np.arange(2 * K), np.arange(4 * K)
    tp = m["target"][:: len(m["target"]) // (2 * K)][: 2 * K]
    mk = lambda d: core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, d, True, ids, tp)
    props = [mk(1), mk(0)]
    comps = [dict(kind=0, weight=0.45, proposal=props[0]), dict(kind=0, weight=0.45, proposal=props[1]), dict(kind=1, weight=0.1, sd=0.1)]
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, 0, True, 0.0, 2.0, 0.0, eids, tp)
    C, n = 64, 200
    th0 = random_theta(m, np.random.default_rng(16), C, alpha_sd=0.3)
    ch = core.Chain(model, tgt, comps, ev, max_chains=C)
    ch.set_statistics(50, 5, 0)
    run = ch.run(th0, n, seed=21)
    assert run["n_accepted"].sum() > C
    sel = _selected(n, 50, 5, 0)
    got = ch.statistics(-1)
    assert got["n"] == C * len(sel)
    _assert_maps(got, core.posterior_variability(model, run["theta"][sel].reshape(-1, K + 10), True))
    for c in (0, 37, 63):
        _assert_maps(ch.statistics(c, False), core.posterior_variability(model, run["theta"][sel, c], False))
    ch.close(); ev.close(); [p.close() for p in props]; model.close(); tgt.close()


def test_face_sized_shape(ctx):
    """N = 28 561 (the face-sized config-5 surface), a few chains and steps, against icp_posterior_variability."""
    m = synth.face_twin(rank=100, side=169)
    tv, tc, _ = synth.partial_target(m, seed=7, alpha_sd=0.5)
    N = len(m["ref"])
    assert N == 28561
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, tv, tc)
    rng = np.random.default_rng(17)
    ids = np.sort(rng.choice(N, 500, replace=False))
    tp = tv[np.sort(rng.choice(len(tv), 500, replace=False))]
    gp = core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, 0, True, ids, tp)
    pose = [dict(kind=2, weight=0.05, sd=0.01, axis=a) for a in range(3)] + [dict(kind=3, weight=0.05, sd=0.1, axis=a) for a in range(3)]
    comps = [dict(kind=0, weight=0.6, proposal=gp), dict(kind=1, weight=0.1, sd=0.05)] + pose
    ev = core.Evaluator(model, tgt, _lib.EVAL_COLLECTIVE, _lib.SYMMETRIC, True, 0.1, 0.3, 1.0, ids, tp)
    C, n = 3, 16
    th0 = random_theta(m, rng, C, alpha_sd=0.3)
    ch = core.Chain(model, tgt, comps, ev, max_chains=C)
    ch.set_statistics(0, 1, 0)
    run = ch.run(th0, n, seed=3)
    assert run["n_accepted"].sum() > 0
    _assert_maps(ch.statistics(-1), core.posterior_variability(model, run["theta"].reshape(-1, 110), True))
    _assert_maps(ch.statistics(2, False), core.posterior_variability(model, run["theta"][:, 2], False))
    ch.close(); ev.close(); gp.close(); model.close(); tgt.close()


def test_sharded_pooled_maps_merge(mix):
    """Two chain objects with chain_id_offset sharding, pooled per object and merged through sharding.merge_variability,
    give the maps of one object over all chains."""
    m, model = mix[0], mix[1]
    C, n, half = 6, 40, 4
    th0 = random_theta(m, np.random.default_rng(18), C, alpha_sd=0.4, pose=True)
    ref = th0[0]
    stats = (5, 2, 0)
    one = _chain(mix, C, stats=stats)
    one.run(th0, n, seed=31)
    want = one.statistics(-1, False, ref)
    parts = []
    for lo, hi in ((0, half), (half, C)):
        sh = _chain(mix, hi - lo, stats=stats)
        sh.run(th0[lo:hi], n, seed=31, chain_id_offset=lo)
        got = sh.statistics(-1, False, ref)
        parts.append(sharding.variability_partials(got["n"], got["mean"], got["cov"]))
        sh.close()
    merged = sharding.merge_variability(np.stack(parts), normals=model.vertex_normals(ref)[0])
    assert merged["n"] == want["n"]
    _assert_maps(merged, want)
    one.close()


def test_argument_checks(mix):
    m = mix[0]
    C, n = 2, 10
    th0 = random_theta(m, np.random.default_rng(19), C, alpha_sd=0.4)
    ch = _chain(mix, C)
    with pytest.raises(_lib.IcpCudaError):
        ch.set_statistics(0, 0)                    # take_every_n < 1
    with pytest.raises(_lib.IcpCudaError):
        ch.set_statistics(-1, 1)                   # burn_in < 0
    with pytest.raises(_lib.IcpCudaError):
        ch.statistics(-1)                          # no resident run
    ch.run(th0, n, seed=1)
    with pytest.raises(_lib.IcpCudaError):
        ch.statistics(-1)                          # statistics were off for the resident run
    ch.set_statistics(n, 1)                        # takes effect at the next run from theta0; burn-in past the run: S == 0
    with pytest.raises(_lib.IcpCudaError):
        ch.statistics(-1)                          # still the run without statistics
    ch.run(th0, n, seed=1)
    with pytest.raises(_lib.IcpCudaError):
        ch.statistics(0)                           # S == 0
    ch.set_statistics(n - 1, 1000, normals=False)  # one sample per chain
    run = ch.run(th0, n, seed=1)
    for bad in (C, -2):
        with pytest.raises(_lib.IcpCudaError):
            ch.statistics(bad)
    with pytest.raises(_lib.IcpCudaError):
        ch.statistics(0, sum_normals=True)         # normals were not accumulated
    one = ch.statistics(0, sum_normals=False)
    assert one["n"] == 1 and np.isnan(one["total_variance"]).all() and np.isnan(one["normal_variance"]).all()
    np.testing.assert_allclose(one["mean"], ch.model.reconstruct(run["theta"][n - 1, 0])[0], rtol=1e-12, atol=1e-10)
    pooled = ch.statistics(-1, sum_normals=False)
    assert pooled["n"] == C and np.isfinite(pooled["total_variance"]).all()
    ch.close()


def test_sampling_registration_variability(ctx, twin31):
    """SamplingRegistration.runfitting(variability=...) leaves the pooled or per-chain maps in self.variability."""
    m = twin31
    model = api.StatisticalMeshModel(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    target = api.TriangleMesh3D(ctx, m["target"], m["target_cells"])
    K = model.rank
    icp = api.MixedProposalDistributions.mixedProposalICP(model, target, 2 * K)
    rnd = api.MixedProposalDistributions.mixedRandomShapeProposal(model)
    gen = api.MixtureProposal.fromProposalsWithTransition((0.9, icp), (0.1, rnd))
    evs = api.ProductEvaluators.proximityAndIndependent(model, target, api.ModelToTargetEvaluation, 2.0, 4 * K)
    reg = api.SamplingRegistration(model, target)
    th0 = np.tile(model.initial_parameters().allParameters, (3, 1))
    th0[1:, 10:] = np.random.default_rng(0).normal(0, 0.3, (2, K))
    var = dict(takeEveryN=5, total=80, burnIn=10, sumNormals=True)
    reg.runfitting(evs, gen, 100, n_chains=3, initial_batch=th0, variability=var)
    pooled = reg.variability
    log = reg.last_run["theta"]
    sel = _selected(100, 10, 5, 80)
    assert pooled["n"] == 3 * len(sel)
    _assert_maps(pooled, core.posterior_variability(model, log[sel].reshape(-1, K + 10), True))
    reg.runfitting(evs, gen, 100, n_chains=3, initial_batch=th0, variability=dict(var, perChain=True, sumNormals=False))
    assert isinstance(reg.variability, list) and len(reg.variability) == 3
    for c, v in enumerate(reg.variability):
        _assert_maps(v, core.posterior_variability(model, reg.last_run["theta"][sel, c], False))
    model.close(); target.close()
