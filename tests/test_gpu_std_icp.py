"""icp_std_icp_*: IcpBasedSurfaceFitting.runfitting (api/other/IcpBasedSurfaceFitting.scala:46-126) for batches of fits on the
device, against the per-call iteration (icp_std_icp_iteration[_theta]) row by row, against the oracle, and for batch / shard
independence, the Philox coin, the failure semantics of :94-104 and the argument checks."""
import numpy as np
import pytest

from conftest import random_theta
from icp_proposal_b200 import _lib, api, core, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

SIGMA2 = (1.0, 0.1, 1e-15)


def _femur(femur, which):
    return dict(ref=femur["ref"], cells=femur["cells"], target=femur["target"], target_cells=femur["target_cells"], **femur[which])


@pytest.fixture(scope="module")
def config2(ctx, femur):
    """Femur GPMM-50 with the point lists of BASELINE config 2 (IcpRegistration.scala:40-43), plus GPMM-100 / GPMM-200."""
    N = 1622
    rng = np.random.default_rng(1024)
    ids = rng.integers(0, N, N)
    tp = synth.near_surface_queries(femur["target"], femur["target_cells"], N, seed=1024, sd=0.0)
    tgt = core.Target(ctx, femur["target"], femur["target_cells"])
    models = {}
    for k in ("50", "100", "200"):
        m = _femur(femur, f"gpmm_{k}")
        models[k] = (core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), m)
    yield dict(ids=ids, tp=tp, tgt=tgt, models=models)
    for model, _ in models.values():
        model.close()
    tgt.close()


def _theta0(m, rng, C, pose):
    th = random_theta(m, rng, C, alpha_sd=0.3, pose=pose)
    if not pose:
        th[:, 7:10] = 0.0   # the identity pose of icp_std_icp_iteration, bit for bit
    return th


def _per_call_rows(model, tgt, ids, tp, th0, sigma2, num_iterations, dirs, log_alpha, pose):
    """Each row of the runner's log from the previous row by the per-call iteration (row -1: theta0)."""
    K = model.K
    want = np.empty_like(log_alpha)
    for it in range(len(log_alpha)):
        s2 = sigma2[it // (num_iterations + 1)]
        prev = th0[:, 10:] if it == 0 else log_alpha[it - 1]
        for d in (0, 1):
            cs = np.nonzero(dirs[it] == d)[0]
            if len(cs) == 0:
                continue
            if pose:
                th = th0[cs].copy()
                th[:, 10:] = prev[cs]
                want[it, cs] = core.std_icp_iteration_theta(model, tgt, d, ids, tp, s2, 1.0, th)
            else:
                want[it, cs] = core.std_icp_iteration(model, tgt, d, ids, tp, s2, 1.0, prev[cs].reshape(-1, K))
    return want


def _assert_rows_close(got, want):
    # the two paths differ in summation order only (projector vs explicit posterior; grouped target observations)
    tol = 1e-8 * np.abs(want).max() + 1e-10
    assert np.abs(got - want).max() <= tol, (np.abs(got - want).max(), tol)


@pytest.mark.parametrize("pose", [False, True])
@pytest.mark.parametrize("mode", ["model", "target", "mixed"])
def test_runner_matches_per_call_loop(config2, mode, pose):
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    C, n_it = 3, 4
    iters = len(SIGMA2) * (n_it + 1)
    rng = np.random.default_rng(7)
    th0 = _theta0(m, rng, C, pose)
    if mode == "mixed":   # per-fit directions that differ between the fits
        dirs = rng.integers(0, 2, (iters, C)).astype(np.int32)
        assert (dirs != dirs[:, :1]).any()
    else:
        dirs = np.full((iters, C), 0 if mode == "model" else 1, np.int32)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_SAMPLING, max_fits=C)
    out = runner.run(th0, SIGMA2, n_it, directions=dirs)
    assert np.array_equal(out["log_direction"], dirs)
    assert (out["status"] == 0).all() and (out["iterations_done"] == iters).all()
    assert np.array_equal(out["alpha_final"], out["log_alpha"][-1])
    want = _per_call_rows(model, tgt, ids, tp, th0, SIGMA2, n_it, dirs, out["log_alpha"], pose)
    _assert_rows_close(out["log_alpha"], want)
    ms, launches = runner.last_run_stats()
    assert ms > 0 and launches >= 5 * iters
    runner.close()


def test_runner_against_oracle(ctx, femur, config2):
    """The first 8 iterations of config 2 against the oracle at the config-2 tolerance."""
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    om = orc.Model(m["ref"], m["cells"], m["basis"], m["variance"])
    ot = orc.Mesh(m["target"], m["target_cells"])
    dirs = np.array([0, 1, 0, 0, 1, 1, 0, 1], np.int32).reshape(-1, 1)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=1)
    out = runner.run(model.theta(center=(0, 0, 0)), (1e-15,), len(dirs) - 1, directions=dirs)
    alpha_o = np.zeros(model.K)
    for it, d in enumerate(dirs[:, 0]):
        alpha_o = orc.std_icp_iteration(om, ot, int(d), ids, tp, 1e-15, 1.0, alpha_o)
        np.testing.assert_allclose(out["log_alpha"][it, 0], alpha_o, rtol=1e-5, atol=1e-6)
    runner.close()


def _coin(ctx, seed, fit, it):
    r = ctx.philox(seed, fit, it, 0)
    u = ((int(r[0]) >> 5) * 67108864 + (int(r[1]) >> 6)) / 9007199254740992.0
    return 0 if u < 0.5 else 1


@pytest.mark.parametrize("k,C,direction", [("50", 37, _lib.MODEL_AND_TARGET_SAMPLING), ("50", 300, _lib.MODEL_AND_TARGET_SAMPLING),
                                           ("50", 37, _lib.MODEL_SAMPLING), ("50", 37, _lib.TARGET_SAMPLING),
                                           ("100", 37, _lib.MODEL_AND_TARGET_SAMPLING), ("200", 9, _lib.MODEL_AND_TARGET_SAMPLING)])
def test_batch_and_shard_independence(ctx, config2, k, C, direction):
    """Fit c of a batch equals the fit run alone (bit for bit); a shard [a, C) with fit_id_offset a equals the second half of
    the full run; run_device equals run. K = 201 takes the large-rank posterior path in target sampling."""
    import torch
    model, m = config2["models"][k]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    n_it, sig = 2, (0.1, 1e-15)
    th0 = _theta0(m, np.random.default_rng(11), C, pose=True)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, direction, max_fits=C)
    full = runner.run(th0, sig, n_it, seed=5)
    assert (full["status"] == 0).all()
    for c in sorted({0, 1, C // 2, C - 1}):
        one = runner.run(th0[c:c + 1], sig, n_it, seed=5, fit_id_offset=c)
        assert np.array_equal(one["log_alpha"][:, 0], full["log_alpha"][:, c])
        assert np.array_equal(one["log_direction"][:, 0], full["log_direction"][:, c])
    a = C // 2
    shard = runner.run(th0[a:], sig, n_it, seed=5, fit_id_offset=a)
    assert np.array_equal(shard["log_alpha"], full["log_alpha"][:, a:])
    assert np.array_equal(shard["alpha_final"], full["alpha_final"][a:])
    # the device entry point
    dev = torch.device("cuda", ctx.device)
    iters = len(sig) * (n_it + 1)
    t0 = torch.tensor(th0, dtype=torch.float64, device=dev)
    fin = torch.empty((C, model.K), dtype=torch.float64, device=dev)
    log = torch.empty((iters, C, model.K), dtype=torch.float64, device=dev)
    ldir, st, done = (torch.zeros(s, dtype=torch.int32, device=dev) for s in ((iters, C), (C,), (C,)))
    torch.cuda.synchronize()
    runner.run_device(C, t0.data_ptr(), sig, n_it, seed=5, alpha_final=fin.data_ptr(), log_alpha=log.data_ptr(),
                      log_direction=ldir.data_ptr(), status=st.data_ptr(), iterations_done=done.data_ptr())
    assert np.array_equal(log.cpu().numpy(), full["log_alpha"])
    assert np.array_equal(fin.cpu().numpy(), full["alpha_final"])
    assert np.array_equal(ldir.cpu().numpy(), full["log_direction"])
    assert (done.cpu().numpy() == iters).all() and (st.cpu().numpy() == 0).all()
    # caller directions in device memory
    dd = torch.tensor(full["log_direction"], dtype=torch.int32, device=dev)
    runner.run_device(C, t0.data_ptr(), sig, n_it, directions=dd.data_ptr(), seed=99, log_alpha=log.data_ptr())
    assert np.array_equal(log.cpu().numpy(), full["log_alpha"])
    runner.close()


def test_philox_coin(ctx, config2):
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    C, n_it, seed, off = 5, 3, 77, 1000
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=C)
    th0 = _theta0(m, np.random.default_rng(3), C, pose=False)
    a = runner.run(th0, (1.0, 1e-15), n_it, seed=seed, fit_id_offset=off)
    b = runner.run(th0, (1.0, 1e-15), n_it, seed=seed, fit_id_offset=off)
    assert np.array_equal(a["log_direction"], b["log_direction"]) and np.array_equal(a["log_alpha"], b["log_alpha"])
    want = np.array([[_coin(ctx, seed, off + c, it) for c in range(C)] for it in range(len(a["log_direction"]))])
    assert np.array_equal(a["log_direction"], want)
    assert set(np.unique(want)) == {0, 1}
    other = runner.run(th0, (1.0, 1e-15), n_it, seed=seed + 1, fit_id_offset=off)
    assert not np.array_equal(other["log_direction"], a["log_direction"])
    runner.close()


def test_failed_fit_keeps_its_coefficients(config2):
    """:94-104: a fit whose coefficients are not finite stops; the others are bit-identical to a run without it."""
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    n_it, sig = 2, (1.0, 1e-15)
    iters = len(sig) * (n_it + 1)
    th0 = _theta0(m, np.random.default_rng(5), 3, pose=True)
    bad = th0[1].copy()
    bad[10 + 4] = np.nan
    th_all = np.stack([th0[0], bad, th0[1], th0[2]])
    dirs = np.random.default_rng(6).integers(0, 2, (iters, 4)).astype(np.int32)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_SAMPLING, max_fits=4)
    got = runner.run(th_all, sig, n_it, directions=dirs)
    ref = runner.run(th0, sig, n_it, directions=dirs[:, [0, 2, 3]])
    assert got["status"][1] & _lib.STD_ICP_NON_FINITE
    assert got["iterations_done"][1] == 0
    for it in range(iters):
        np.testing.assert_array_equal(got["log_alpha"][it, 1], bad[10:])   # NaN in the same place, the rest unchanged
    np.testing.assert_array_equal(got["alpha_final"][1], bad[10:])
    assert np.array_equal(got["log_alpha"][:, [0, 2, 3]], ref["log_alpha"])
    assert (got["status"][[0, 2, 3]] == 0).all() and (got["iterations_done"][[0, 2, 3]] == iters).all()
    runner.close()


def test_config2_in_full(config2, femur):
    """Config 2: one fit, 101 iterations at sigma2 = 1e-15, alternating directions."""
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    dirs = (np.arange(101) % 2).astype(np.int32).reshape(-1, 1)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=1)
    out = runner.run(model.theta(center=(0, 0, 0)), (1e-15,), 100, directions=dirs)
    assert out["status"][0] == 0 and out["iterations_done"][0] == 101
    dist = np.sqrt(tgt.closest_point_surface(model.reconstruct(model.theta(out["alpha_final"][0], center=(0, 0, 0)))[0])[3])
    d0 = np.sqrt(tgt.closest_point_surface(m["ref"])[3])
    assert dist.mean() < 1.0 and dist.mean() < 0.2 * d0.mean()
    runner.close()


@pytest.mark.parametrize("direction", [0, 1])
def test_open_surface(ctx, open_twin, direction):
    m = open_twin
    model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt = core.Target(ctx, m["target"], m["target_cells"])
    assert tgt.boundary_flags().any()
    ids = np.arange(0, len(m["ref"]), 3)
    tp = m["target"][::2]
    C, n_it, sig = 2, 3, (1.0, 1e-3)
    th0 = _theta0(m, np.random.default_rng(8), C, pose=True)
    dirs = np.full((len(sig) * (n_it + 1), C), direction, np.int32)
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, direction, max_fits=C)
    out = runner.run(th0, sig, n_it)
    assert np.array_equal(out["log_direction"], dirs)
    _assert_rows_close(out["log_alpha"], _per_call_rows(model, tgt, ids, tp, th0, sig, n_it, dirs, out["log_alpha"], True))
    runner.close(); model.close(); tgt.close()


def test_api_batched_initial_coefficients(ctx, config2):
    _, m = config2["models"]["50"]
    model = api.StatisticalMeshModel(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    C, n_it, sig = 3, 2, (1.0, 1e-15)
    iters = len(sig) * (n_it + 1)
    alpha0 = np.random.default_rng(9).normal(0, 0.3, (C, model.K))
    dirs = np.where(np.random.default_rng(10).random((iters, C)) < 0.5, api.ModelSampling, api.TargetSampling)
    fit = api.IcpBasedSurfaceFitting(model, tgt, len(ids), 1.0, api.ModelAndTargetSampling, model_point_ids=ids, target_points=tp)
    meshes = fit.runfitting(n_it, sig, initialCoefficients=alpha0, directions=dirs)
    assert len(meshes) == C and fit.coefficients.shape == (C, model.K)
    for c in range(C):
        one = api.IcpBasedSurfaceFitting(model, tgt, len(ids), 1.0, api.ModelAndTargetSampling, model_point_ids=ids, target_points=tp)
        mesh = one.runfitting(n_it, sig, initialCoefficients=alpha0[c], directions=list(dirs[:, c]))
        assert np.array_equal(one.coefficients, fit.coefficients[c])
        assert np.array_equal(mesh, meshes[c])
    model.close()


def test_argument_checks_and_references(ctx, config2):
    model, m = config2["models"]["50"]
    tgt, ids, tp = config2["tgt"], config2["ids"], config2["tp"]
    lib = model.lib
    bad_ids = ids.copy(); bad_ids[3] = model.N
    with pytest.raises(_lib.IcpCudaError):
        core.StdIcp(model, tgt, bad_ids, tp)
    with pytest.raises(_lib.IcpCudaError):
        core.StdIcp(model, tgt, ids, tp, direction=3)
    with pytest.raises(_lib.IcpCudaError):                   # only the runner accepts ModelAndTargetSampling
        core.IcpProposal(model, tgt, 0.1, 10.0, 5.0, _lib.MODEL_AND_TARGET_SAMPLING, False, ids, tp)
    ctx2 = core.Context(ctx.device)
    tgt2 = core.Target(ctx2, m["target"], m["target_cells"])
    with pytest.raises(_lib.IcpCudaError):
        core.StdIcp(model, tgt2, ids, tp)
    tgt2.close(); ctx2.close()
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_AND_TARGET_SAMPLING, max_fits=2)
    th0 = np.stack([model.theta(center=(0, 0, 0))] * 3)
    for args, kw in [((th0, (1.0,), 1), {}),                                    # C > max_fits
                     ((th0[:2], (), 1), {}),                                   # n_sigma < 1
                     ((th0[:2], (0.0,), 1), {}), ((th0[:2], (np.nan,), 1), {}), ((th0[:2], (-1.0,), 1), {}),
                     ((th0[:2], (1.0,), -1), {}),
                     ((th0[:2], (1.0,), 1), dict(directions=np.full((2, 2), 2)))]:
        with pytest.raises(_lib.IcpCudaError) as e:
            runner.run(*args, **kw)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    io = _lib.StdIcpIO()
    assert lib.icp_std_icp_run(runner.h, 0, _lib.dptr(th0), 1, _lib.dptr(np.ones(1)), 1, io) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_std_icp_run(runner.h, 1, None, 1, _lib.dptr(np.ones(1)), 1, io) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_std_icp_run(None, 1, _lib.dptr(th0), 1, _lib.dptr(np.ones(1)), 1, io) == _lib.ERR_INVALID_ARGUMENT
    # the handle holds references: the model and the target cannot go while it lives
    assert lib.icp_model_destroy(model.h) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_target_destroy(tgt.h) == _lib.ERR_INVALID_ARGUMENT
    out = runner.run(th0[:2], (1.0,), 1)                      # and the handle still works
    assert (out["status"] == 0).all()
    runner.close()
