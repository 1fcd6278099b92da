"""Registration measures and the Dice coefficient over a target set (icp_registration_metrics_targets /
icp_dice_coefficient_targets): every row equals, bit for bit, the single-target call on its own target, for targets of
different vertex counts, sets with an open target, caller and seeded Dice samples, calls that span several chunks, NaN rows;
the oracle on a few rows; the argument checks and the host layers."""
import numpy as np
import pytest

from icp_proposal_b200 import _lib, api, core, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

K = 101
# rows per chunk of the target-set calls (csrc/metrics.cu, DESIGN.md section 5)
METRICS_CHUNK_POINTS, DICE_CHUNK_POINTS = 1 << 23, 1 << 25


def _base(femur):
    return dict(ref=femur["ref"], cells=femur["cells"], **femur["gpmm_100"])


def _perturbed(base, t_index):
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


def _thetas(model, rng, n, alpha_sd=0.5):
    th = np.stack([model.theta(rng.normal(0, alpha_sd, K)) for _ in range(n)])
    th[:, 1:4] = rng.normal(0, 1.0, (n, 3))
    th[:, 4:7] = rng.normal(0, 0.02, (n, 3))
    return th


class Targets:
    def __init__(self, ctx, femur, open_target=False):
        base = _base(femur)
        self.model = core.Model(ctx, base["ref"], base["cells"], base["basis"], base["variance"])
        self.meshes = [_perturbed(base, 0), _split_centroids(*_perturbed(base, 2), 40), _perturbed(base, 1)]
        if open_target:
            tv, tc, _ = synth.partial_target(base, seed=5, alpha_sd=0.3)
            self.meshes[2] = (tv, tc)
        self.targets = [core.Target(ctx, v, c) for v, c in self.meshes]

    def close(self):
        for t in self.targets:
            t.close()
        self.model.close()


def _single(fn, model, targets, th, tidx, **kw):
    """Row c of the single-target call on targets[tidx[c]] (each target's rows in one call: the rows are independent)."""
    out = None
    for g in np.unique(tidx):
        rows = np.flatnonzero(tidx == g)
        got = fn(model, targets[g], th[rows], **kw)
        if out is None:
            out = np.empty((len(th),) + got.shape[1:])
        out[rows] = got
    return out


def _equal(a, b):
    return np.array_equal(a, b, equal_nan=True)


@pytest.fixture(scope="module")
def closed(ctx, femur):
    s = Targets(ctx, femur)
    yield s
    s.close()


@pytest.fixture(scope="module")
def with_open(ctx, femur):
    s = Targets(ctx, femur, open_target=True)
    yield s
    s.close()


def test_three_targets_of_different_vertex_counts(closed):
    """An unsorted, non-contiguous index over targets of 1622, 1662 and 1622 vertices, one of them listed twice."""
    S = closed
    assert len(S.meshes[1][0]) == len(S.meshes[0][0]) + 40
    targets = S.targets + [S.targets[0]]
    th = _thetas(S.model, np.random.default_rng(3), 11)
    tidx = np.array([2, 0, 3, 1, 1, 2, 0, 3, 1, 2, 0])
    got = core.registration_metrics(S.model, targets, th, target_index=tidx)
    want = _single(core.registration_metrics, S.model, targets, th, tidx)
    assert _equal(got, want)
    assert np.all(np.isfinite(got)) and len(np.unique(got[:, 1])) == len(th)
    assert np.array_equal(got[:, 0], got[:, 2]) and np.all(got[:, 3] <= got[:, 1])   # closed targets: no filter


def test_boundary_set(with_open):
    """An open target in the set: every row takes the boundary filter, a closed target's rows still equal their plain call."""
    S = with_open
    assert S.targets[2].boundary_flags().any() and not S.targets[0].boundary_flags().any()
    th = _thetas(S.model, np.random.default_rng(5), 9)
    tidx = np.array([2, 1, 0, 2, 0, 1, 2, 2, 0])
    got = core.registration_metrics(S.model, S.targets, th, target_index=tidx)
    want = _single(core.registration_metrics, S.model, S.targets, th, tidx)
    assert _equal(got, want)
    op = tidx == 2
    assert np.all(got[op, 2] != got[op, 0])                          # the filter dropped something on the open target
    assert np.array_equal(got[~op, 0], got[~op, 2])


def test_dice_bit_for_bit_and_against_the_oracle(ctx, femur, closed):
    S = closed
    rng = np.random.default_rng(9)
    th = _thetas(S.model, rng, 7, alpha_sd=0.3)
    th[4, 1] += 15.0                                                 # a clearly displaced mesh: lower overlap
    tidx = np.array([1, 0, 2, 1, 1, 0, 2])
    u = rng.random((4000, 3))
    got = core.dice_coefficient(S.model, S.targets, th, unit_samples=u, target_index=tidx)
    assert _equal(got, _single(core.dice_coefficient, S.model, S.targets, th, tidx, unit_samples=u))
    seeded = core.dice_coefficient(S.model, S.targets, th, n_samples=10000, seed=7, target_index=tidx)
    assert _equal(seeded, _single(core.dice_coefficient, S.model, S.targets, th, tidx, n_samples=10000, seed=7))
    assert got[4] < got[0] - 0.05 and np.all((0 < got) & (got <= 1))
    assert np.all(np.abs(seeded - got) < 0.05)
    # the oracle on a few rows, with the tolerances of the single-target tests
    base = _base(femur)
    om = orc.Model(base["ref"], base["cells"], base["basis"], base["variance"])
    metrics = core.registration_metrics(S.model, S.targets, th, target_index=tidx)
    for c in (0, 2, 4):
        ot = orc.Mesh(*S.meshes[tidx[c]])
        assert abs(got[c] - orc.dice_coefficient(om, ot, th[c], u)) <= 2.0 * 2 / 4000
        np.testing.assert_allclose(metrics[c], orc.registration_metrics(om, ot, th[c]), rtol=1e-9)


def test_calls_spanning_several_chunks(with_open):
    S = with_open
    rng = np.random.default_rng(13)
    N, max_nt = S.model.N, max(len(v) for v, _ in S.meshes)
    rows = METRICS_CHUNK_POINTS // (N + max_nt)
    C = rows + 37
    th = _thetas(S.model, rng, C)
    tidx = rng.integers(0, 3, C)
    got = core.registration_metrics(S.model, S.targets, th, target_index=tidx)
    assert _equal(got, _single(core.registration_metrics, S.model, S.targets, th, tidx))
    n = (1 << 23) + 1
    assert DICE_CHUNK_POINTS // n == 3                               # 4 rows: chunks of 3 and 1
    th4, tidx4 = th[:4], np.array([1, 0, 2, 0])
    got = core.dice_coefficient(S.model, S.targets, th4, n_samples=n, seed=3, target_index=tidx4)
    assert _equal(got, _single(core.dice_coefficient, S.model, S.targets, th4, tidx4, n_samples=n, seed=3))


def test_edge_cases(closed):
    S = closed
    th = _thetas(S.model, np.random.default_rng(17), 5)
    th[3, 12] = np.nan
    one = core.registration_metrics(S.model, S.targets[1], th)
    assert np.isnan(one[3, 0]) and np.all(np.isfinite(np.delete(one, 3, 0)))
    assert _equal(core.registration_metrics(S.model, [S.targets[1]], th), one)
    assert _equal(core.registration_metrics(S.model, [S.targets[1]], th, target_index=np.zeros(5)), one)
    tidx = np.array([0, 2, 1, 1, 0])
    assert _equal(core.registration_metrics(S.model, S.targets, th, target_index=tidx),
                  _single(core.registration_metrics, S.model, S.targets, th, tidx))
    d1 = core.dice_coefficient(S.model, S.targets[1], th, n_samples=2000, seed=5)
    assert _equal(core.dice_coefficient(S.model, [S.targets[1]], th, n_samples=2000, seed=5), d1)
    assert _equal(core.dice_coefficient(S.model, S.targets, th, n_samples=2000, seed=5, target_index=tidx),
                  _single(core.dice_coefficient, S.model, S.targets, th, tidx, n_samples=2000, seed=5))
    assert core.registration_metrics(S.model, S.targets, th[:0], target_index=tidx[:0]).shape == (0, 4)
    assert core.dice_coefficient(S.model, S.targets, th[:0], target_index=tidx[:0]).shape == (0,)


def test_argument_checks(ctx, femur, closed):
    S = closed
    th = _thetas(S.model, np.random.default_rng(19), 3)

    def refused(match, targets, tidx, dice=False):
        fn = core.dice_coefficient if dice else core.registration_metrics
        with pytest.raises(_lib.IcpCudaError, match=match) as e:
            fn(S.model, targets, th, target_index=tidx)
        assert e.value.code == _lib.ERR_INVALID_ARGUMENT

    for dice in (False, True):
        refused(r"target_index\[1\] = 3 is outside \[0, n_targets\)", S.targets, [0, 3, 1], dice)
        refused(r"target_index\[2\] = -1 is outside", S.targets, [0, 1, -1], dice)
        refused("target_index is required when n_targets > 1", S.targets, None, dice)
        gone = core.Target(ctx, *S.meshes[0])
        gone.close()
        refused(r"targets\[1\] is null", [S.targets[0], gone], [0, 0, 0], dice)
        other = core.Context(0)
        foreign = core.Target(other, *S.meshes[0])
        refused(r"targets\[2\] belongs to another context", [S.targets[0], S.targets[1], foreign], [0, 0, 0], dice)
        foreign.close(); other.close()
    # the refused calls left nothing behind: a valid call still gives the single-target rows
    tidx = np.array([1, 0, 1])
    assert _equal(core.registration_metrics(S.model, S.targets, th, target_index=tidx),
                  _single(core.registration_metrics, S.model, S.targets, th, tidx))


def test_registration_comparison_over_a_target_set(closed):
    S = closed
    th = _thetas(S.model, np.random.default_rng(23), 6)
    tidx = np.array([2, 2, 0, 1, 0, 1])
    params = [api.ModelFittingParameters.from_vector(t) for t in th]
    metrics = api.RegistrationComparison.evaluateReconstructions2GroundTruth(S.model, params, S.targets, tidx)
    for c in range(len(th)):
        assert _equal(metrics[c], core.registration_metrics(S.model, S.targets[tidx[c]], th[c:c + 1])[0])
    m2, dice = api.RegistrationComparison.evaluateReconstructions2GroundTruth(S.model, th, S.targets, tidx, dice=True,
                                                                                n_samples=3000, seed=11)
    assert _equal(m2, metrics)
    for c in range(len(th)):
        assert _equal(dice[c:c + 1], core.dice_coefficient(S.model, S.targets[tidx[c]], th[c:c + 1], n_samples=3000, seed=11))
