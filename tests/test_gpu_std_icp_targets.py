"""Deterministic-ICP handles over several targets (icp_std_icp_create_targets / icp_std_icp_set_target_index): every fit of
a multi-target run equals the single-target run of that fit on its own target, bit for bit, in both directions, with the
Philox coin and with caller directions, through sharded and device runs; the oracle per target; targets of different vertex
counts and open targets; the failure semantics; api.IcpBasedSurfaceFitting.runfittings; the argument checks."""
import numpy as np
import pytest

from conftest import random_theta
from icp_proposal_b200 import _lib, api, core, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

N_PTS = 400
KEYS = ("alpha_final", "log_alpha", "log_direction", "status", "iterations_done")
SIG = (0.1, 1e-15)


def _perturbed(femur, t_index):
    """Perturbed femur-twin targets (GPMM-100 instances plus vertex noise), as in tests/test_gpu_multi_target.py."""
    base = dict(ref=femur["ref"], **femur["gpmm_100"])
    target = synth.model_instance(base, np.random.default_rng(100 + t_index).normal(0, 1.0, len(base["variance"])))
    return target + np.random.default_rng(7 + t_index).normal(0, 0.5, target.shape), femur["cells"]


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
    """A model and G targets, each with its own target-surface point list of n_tp points."""

    def __init__(self, ctx, m, meshes, n_ids=N_PTS, n_tp=N_PTS, seed=1):
        self.m = m
        self.model = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
        self.meshes = meshes
        self.targets = [core.Target(ctx, tv, tc) for tv, tc in meshes]
        self.tps = [synth.near_surface_queries(tv, tc, n_tp, seed=seed + g, sd=0.0) for g, (tv, tc) in enumerate(meshes)]
        self.ids = np.random.default_rng(seed).integers(0, len(m["ref"]), n_ids)

    def multi(self, C, direction=_lib.MODEL_AND_TARGET_SAMPLING):
        return core.StdIcp(self.model, model_point_ids=self.ids, direction=direction, max_fits=C,
                           targets=list(zip(self.targets, self.tps)))

    def single(self, g, C=1, direction=_lib.MODEL_AND_TARGET_SAMPLING):
        return core.StdIcp(self.model, self.targets[g], self.ids, self.tps[g], 1.0, direction, max_fits=C)

    def theta0(self, C, seed, pose=True):
        th = random_theta(self.m, np.random.default_rng(seed), C, alpha_sd=0.3, pose=pose)
        if not pose:
            th[:, 7:10] = 0.0
        return th

    def close(self):
        for t in self.targets:
            t.close()
        self.model.close()


def _model(femur, k):
    return dict(ref=femur["ref"], cells=femur["cells"], **femur[f"gpmm_{k}"])


@pytest.fixture(scope="module")
def sets(ctx, femur):
    """GPMM-50 and GPMM-200 of the femur against three perturbed femur-twin targets."""
    meshes = [_perturbed(femur, t) for t in range(3)]
    out = {k: Set(ctx, _model(femur, k), meshes) for k in ("50", "200")}
    yield out
    for s in out.values():
        s.close()


def _fit_of(out, c):
    return {k: (out[k][:, c] if k in ("log_alpha", "log_direction") else out[k][c]) for k in KEYS}


def _assert_fits_equal_singles(S, multi, th0, tidx, n_it, seed, off, dirs=None, direction=_lib.MODEL_AND_TARGET_SAMPLING, sig=SIG):
    singles = {}
    for c in range(len(th0)):
        g = int(tidx[c])
        if g not in singles:
            singles[g] = S.single(g, direction=direction)
        one = singles[g].run(th0[c:c + 1], sig, n_it, seed=seed, fit_id_offset=off + c,
                             directions=None if dirs is None else dirs[:, c:c + 1])
        a, b = _fit_of(multi, c), _fit_of(one, 0)
        for k in KEYS:
            assert np.array_equal(a[k], b[k], equal_nan=True), f"{k} of fit {c} (target {g}) differs from its single-target run"
    for r in singles.values():
        r.close()


@pytest.mark.parametrize("k", ["50", "200"])
@pytest.mark.parametrize("pose", [False, True])
@pytest.mark.parametrize("mode", ["model", "target", "philox", "caller"])
def test_fits_equal_their_single_target_runs(sets, k, pose, mode):
    """G = 3, a non-contiguous unsorted target index: every fit's outputs equal those of a single-target handle on its own
    target with the same seed and global fit id. K = 200 takes the large-rank posterior path in target sampling."""
    S = sets[k]
    C, n_it, seed, off = 7, 2, 5, 3
    tidx = np.array([2, 0, 2, 1, 0, 1, 2])
    iters = len(SIG) * (n_it + 1)
    th0 = S.theta0(C, 11, pose)
    direction = {"model": _lib.MODEL_SAMPLING, "target": _lib.TARGET_SAMPLING}.get(mode, _lib.MODEL_AND_TARGET_SAMPLING)
    dirs = np.random.default_rng(12).integers(0, 2, (iters, C)).astype(np.int32) if mode == "caller" else None
    runner = S.multi(C, direction)
    out = runner.run(th0, SIG, n_it, seed=seed, fit_id_offset=off, directions=dirs, target_index=tidx)
    runner.close()
    assert (out["status"] == 0).all() and (out["iterations_done"] == iters).all()
    if mode in ("philox", "caller"):
        assert set(np.unique(out["log_direction"])) == {0, 1}
    _assert_fits_equal_singles(S, out, th0, tidx, n_it, seed, off, dirs, direction)


def test_batching_sharding_and_run_device(ctx, sets):
    """The set split into two runs with fit_id_offset, a later run that keeps the target index, and run_device all equal the
    full run bit for bit."""
    import torch
    S = sets["50"]
    C, n_it, seed = 9, 2, 17
    tidx = np.array([1, 1, 0, 2, 0, 2, 2, 1, 0])
    th0 = S.theta0(C, 21)
    runner = S.multi(C)
    full = runner.run(th0, SIG, n_it, seed=seed, target_index=tidx)
    again = runner.run(th0, SIG, n_it, seed=seed)                     # the index is kept for runs with the same C
    for k in KEYS:
        assert np.array_equal(again[k], full[k])
    a = 4
    parts = [runner.run(th0[:a], SIG, n_it, seed=seed, target_index=tidx[:a]),
             runner.run(th0[a:], SIG, n_it, seed=seed, fit_id_offset=a, target_index=tidx[a:])]
    for k in KEYS:
        axis = 1 if k in ("log_alpha", "log_direction") else 0
        assert np.array_equal(np.concatenate([p[k] for p in parts], axis=axis), full[k]), k
    dev = torch.device("cuda", ctx.device)
    iters = len(SIG) * (n_it + 1)
    t0 = torch.tensor(th0, dtype=torch.float64, device=dev)
    fin = torch.empty((C, S.model.K), dtype=torch.float64, device=dev)
    log = torch.empty((iters, C, S.model.K), dtype=torch.float64, device=dev)
    ldir, st, done = (torch.zeros(s, dtype=torch.int32, device=dev) for s in ((iters, C), (C,), (C,)))
    torch.cuda.synchronize()
    runner.run_device(C, t0.data_ptr(), SIG, n_it, seed=seed, alpha_final=fin.data_ptr(), log_alpha=log.data_ptr(),
                      log_direction=ldir.data_ptr(), status=st.data_ptr(), iterations_done=done.data_ptr(), target_index=tidx)
    assert np.array_equal(log.cpu().numpy(), full["log_alpha"])
    assert np.array_equal(fin.cpu().numpy(), full["alpha_final"])
    assert np.array_equal(ldir.cpu().numpy(), full["log_direction"])
    assert np.array_equal(st.cpu().numpy(), full["status"]) and np.array_equal(done.cpu().numpy(), full["iterations_done"])
    runner.close()


def test_oracle_per_target(femur, sets):
    """One fit per target, caller directions: every log row against orc.std_icp_iteration on that fit's own target, applied
    to the runner's previous row, at the tolerance of the single-target oracle test."""
    S = sets["50"]
    m = S.m
    om = orc.Model(m["ref"], m["cells"], m["basis"], m["variance"])
    dirs = np.array([[0, 1, 1], [1, 0, 1], [0, 0, 1], [1, 1, 0], [0, 1, 0], [1, 0, 0]], np.int32)
    tidx = np.array([2, 0, 1])
    th0 = np.stack([S.model.theta(center=(0, 0, 0))] * 3)
    runner = S.multi(3)
    out = runner.run(th0, (1e-15,), len(dirs) - 1, directions=dirs, target_index=tidx)
    runner.close()
    for c, g in enumerate(tidx):
        ot = orc.Mesh(*S.meshes[g])
        prev = np.zeros(S.model.K)
        for it in range(len(dirs)):
            want = orc.std_icp_iteration(om, ot, int(dirs[it, c]), S.ids, S.tps[g], 1e-15, 1.0, prev)
            np.testing.assert_allclose(out["log_alpha"][it, c], want, rtol=1e-5, atol=1e-6)
            prev = out["log_alpha"][it, c]


def test_targets_of_different_vertex_counts(ctx, femur):
    """Closed targets with 1622 and 1622 + 40 vertices (and more triangles) in one set."""
    a = _perturbed(femur, 0)
    b = _split_centroids(*_perturbed(femur, 1), 40)
    S = Set(ctx, _model(femur, "50"), [a, b])
    assert len(b[0]) == len(a[0]) + 40 and len(b[1]) == len(a[1]) + 80
    C, n_it = 6, 2
    tidx = np.array([1, 0, 0, 1, 1, 0])
    th0 = S.theta0(C, 31)
    runner = S.multi(C)
    out = runner.run(th0, SIG, n_it, seed=9, target_index=tidx)
    runner.close()
    assert set(np.unique(out["log_direction"])) == {0, 1}
    _assert_fits_equal_singles(S, out, th0, tidx, n_it, 9, 0)
    S.close()


def test_open_targets(ctx, open_twin):
    """Two partial (open) targets of the open test model: the runner has no boundary filter, so fits stay bit-identical."""
    m = open_twin
    tv2, tc2, _ = synth.partial_target(m, seed=5, alpha_sd=0.4)
    S = Set(ctx, m, [(m["target"], m["target_cells"]), (tv2, tc2)], n_ids=300, n_tp=300)
    assert all(t.boundary_flags().any() for t in S.targets)
    C, n_it = 4, 3
    tidx = np.array([1, 0, 1, 0])
    th0 = S.theta0(C, 41)
    runner = S.multi(C)
    out = runner.run(th0, (1.0, 1e-3), n_it, seed=3, target_index=tidx)
    runner.close()
    _assert_fits_equal_singles(S, out, th0, tidx, n_it, 3, 0, sig=(1.0, 1e-3))
    S.close()


def test_failed_fit_leaves_other_targets_untouched(sets):
    """A fit with a non-finite theta0 on target 1 stops; the fits on every target equal the run without it."""
    S = sets["50"]
    n_it = 2
    iters = len(SIG) * (n_it + 1)
    th0 = S.theta0(5, 51)
    bad = th0[2].copy()
    bad[10 + 3] = np.nan
    th_all = np.concatenate([th0[:2], bad[None], th0[2:]])
    tidx = np.array([0, 2, 1, 1, 0, 2])
    dirs = np.random.default_rng(52).integers(0, 2, (iters, 6)).astype(np.int32)
    keep = [0, 1, 3, 4, 5]
    runner = S.multi(6)
    got = runner.run(th_all, SIG, n_it, directions=dirs, target_index=tidx)
    ref = runner.run(th0, SIG, n_it, directions=dirs[:, keep], target_index=tidx[keep])
    runner.close()
    assert got["status"][2] & _lib.STD_ICP_NON_FINITE and got["iterations_done"][2] == 0
    np.testing.assert_array_equal(got["alpha_final"][2], bad[10:])
    for k in KEYS:
        sel = got[k][:, keep] if k in ("log_alpha", "log_direction") else got[k][keep]
        assert np.array_equal(sel, ref[k]), k
    assert (ref["status"] == 0).all()


def test_api_runfittings_equals_each_runfitting(ctx, sets):
    """Three fittings on three targets (one of them a single fit), ModelAndTargetSampling with the coins of each fitting's
    own rand: each fitting's coefficients and instances equal those of its own runfitting. Fittings that differ in anything
    but the target are refused."""
    S = sets["50"]
    m = S.m
    model = api.StatisticalMeshModel(ctx, m["ref"], m["cells"], m["basis"], m["variance"])
    n_it, sig = 2, (1.0, 1e-15)
    inits = [np.random.default_rng(60).normal(0, 0.3, (3, model.K)), np.random.default_rng(61).normal(0, 0.3, model.K),
             np.random.default_rng(62).normal(0, 0.3, (2, model.K))]

    def fittings(**kw):
        out = []
        for g in range(3):
            a = dict(stepLength=1.0, projectionDirection=api.ModelAndTargetSampling, ids=S.ids)
            a.update(kw if g == 2 else {})
            out.append(api.IcpBasedSurfaceFitting(model, S.targets[g], N_PTS, a["stepLength"], a["projectionDirection"],
                                                  rand=np.random.default_rng(70 + g), model_point_ids=a["ids"],
                                                  target_points=S.tps[g]))
        return out

    batch = fittings()
    got = api.IcpBasedSurfaceFitting.runfittings(batch, n_it, sig, inits)
    for g, one in enumerate(fittings()):
        want = one.runfitting(n_it, sig, initialCoefficients=inits[g])
        assert np.array_equal(batch[g].coefficients, one.coefficients), f"fitting {g}"
        if g == 1:
            assert np.array_equal(got[g], want)
        else:
            assert len(got[g]) == len(want) and all(np.array_equal(x, y) for x, y in zip(got[g], want))
    for kw, field in ((dict(stepLength=0.5), "stepLength"), (dict(projectionDirection=api.ModelSampling), "projectionDirection"),
                      (dict(ids=S.ids[::-1].copy()), "model_point_ids")):
        with pytest.raises(ValueError, match=field):
            api.IcpBasedSurfaceFitting.runfittings(fittings(**kw), n_it, sig, inits)
    model.close()


def test_argument_checks_and_references(ctx, femur):
    meshes = [_perturbed(femur, t) for t in range(2)]
    S = Set(ctx, _model(femur, "50"), meshes)
    model, lib = S.model, S.model.lib
    (t0, t1), (tp0, tp1) = S.targets, S.tps

    def create(ents):
        arr = (_lib.StdIcpTarget * len(ents))()
        for g, (t, tp) in enumerate(ents):
            arr[g].target = t.h if t is not None else None
            arr[g].target_points = _lib.dptr(tp) if tp is not None else None
        h = _lib.C.c_void_p()
        rc = lib.icp_std_icp_create_targets(model.h, len(ents), arr, _lib.iptr(_lib.i32(S.ids)), len(S.ids), len(tp0), 1.0,
                                            _lib.MODEL_AND_TARGET_SAMPLING, 4, _lib.C.byref(h))
        return rc, h

    def refused(ents, what):
        rc, _ = create(ents)
        assert rc == _lib.ERR_INVALID_ARGUMENT
        msg = _lib.last_error(model.ctx.h)
        assert what in msg, msg

    refused([(t0, tp0), (None, tp1)], "targets[1].target")
    refused([(t0, tp0), (t1, None)], "targets[1].target_points")
    nan_tp = tp1.copy(); nan_tp[7, 1] = np.nan
    refused([(t0, tp0), (t1, nan_tp)], "targets[1].target_points must be finite")
    ctx2 = core.Context(ctx.device)
    t_other = core.Target(ctx2, *meshes[1])
    refused([(t0, tp0), (t_other, tp1)], "targets[1].target")
    t_other.close(); ctx2.close()
    with pytest.raises(ValueError, match="target points"):
        core.StdIcp(model, model_point_ids=S.ids, max_fits=4, targets=[(t0, tp0), (t1, tp1[:-1])])

    runner = S.multi(4)
    th0 = S.theta0(3, 1)
    with pytest.raises(_lib.IcpCudaError, match="set_target_index"):
        runner.run(th0, (1.0,), 1)                                                   # no target index yet
    for bad, where in (([0, 2, 1], "target_index[1]"), ([0, 1, -1], "target_index[2]")):
        with pytest.raises(_lib.IcpCudaError, match=r"target_index\[") as e:
            runner.set_target_index(bad)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT and where in str(e.value)
    with pytest.raises(_lib.IcpCudaError) as e:
        runner.set_target_index([0] * 5)                                             # C > max_fits
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    runner.set_target_index([0, 1])
    with pytest.raises(_lib.IcpCudaError, match="set_target_index") as e:
        runner.run(th0, (1.0,), 1)                                                   # the last index had C = 2
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    out = runner.run(th0, (1.0,), 1, target_index=[0, 1, 1])
    assert (out["status"] == 0).all()
    # the handle holds a reference on every target; destroying it releases them
    assert lib.icp_target_destroy(t0.h) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_target_destroy(t1.h) == _lib.ERR_INVALID_ARGUMENT
    assert lib.icp_model_destroy(model.h) == _lib.ERR_INVALID_ARGUMENT
    runner.close()
    S.close()
