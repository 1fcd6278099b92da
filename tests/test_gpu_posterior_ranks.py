"""Every rank-dependent posterior kernel variant, K = 1 to 224, against an extended-precision reference.

The padded rank Kp = 8 ceil(K / 8), the batch size C and the observation count pick the kernels of the posterior:

    FP64 rank update          launch_fused<4,4,4> / <8,7,4> / <24,13,4>   NB = Kp / 8 <= 4 / 5..7 / 8..13
                              launch_pb_mma<28,20,8> / <36,28,12>         NB 14..20 / 21..28
    factorisation             k_cholesky_packed NT = 256 / NT = 128       Kp <= 104 with C <= 148 / C > 148
                              k_cholesky_solve_mma                        104 < Kp <= 160
                              k_pack_lower + k_cholesky_packed            160 < Kp <= 224
    unstaged observation ids  k_posterior_build_mma / k_posterior_fused   more than kMaxStagedIds = 4096 observations
    INT8 rank update          falls back to FP64                          Kp > 112, or n * rows per observation > 32000
    SVD factor                H, J in shared / one in global / both       Kp <= 112 / 120..160 / >= 168
    k_si_project<7/13/28>     std-ICP model sampling                      NB <= 7 / <= 13 / <= 28
    k_chain_propose           packed L in shared memory                   every chain (214 KB at K = 224)
    k_cholesky_solve (+ k_mean_to_ymean), k_posterior_fused<.., true>     ICPCUDA_NO_DMMA=1 / ICPCUDA_FUSE=1

The reference is a Cholesky, triangular solves and a quadratic form in np.longdouble (80-bit, eps ~ 1.1e-19): three
orders of magnitude below the device's rounding, so what the comparison sees is the device's error alone. Tolerances are
functions of K, the unit roundoff u of float64 and the condition number of the matrix, or exact equalities.

Run as a script with --child, the file repeats the factorisation and pipeline checks at four ranks and prints a summary:
the environment-selected paths read their variable once per process, so they run in a child process.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import random_theta  # also puts the repository root on sys.path (script mode)
from icp_proposal_b200 import _lib, core, synth
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

LD = np.longdouble
U = np.finfo(np.float64).eps / 2     # unit roundoff of the device's FP64 arithmetic
STEP = 0.1
SENTINEL = -7.25                     # the upper triangle of L as passed in: the device must leave it alone
RANKS = (1, 8, 9, 32, 33, 56, 57, 104, 105, 112, 113, 160, 161, 168, 169, 223, 224)
# the INT8 split-integer emulation's accuracy on M relative to max|M| (tc_i8.cu), the bound the other INT8 tests use
I8_BOUND = 2e-8
MODES = {   # (direction, sd_t, sd_n): sd_n <= sd_t with every observation kept is the constant-Gram path (one row per
            # observation); sd_n > sd_t the general three-row update
    "model_rpo1": (_lib.MODEL_SAMPLING, 10.0, 5.0),
    "model_rpo3": (_lib.MODEL_SAMPLING, 5.0, 10.0),
    "target": (_lib.TARGET_SAMPLING, 10.0, 5.0),
}


def kp(K):
    return (K + 7) // 8 * 8


def factor_path(K, C):
    """The factorisation icp_debug_factor (and the pipeline) runs at rank K for a batch of C matrices."""
    if kp(K) <= 104:
        return "k_cholesky_packed NT=%d" % (256 if C <= 148 else 128)
    if kp(K) <= 160:
        return "k_cholesky_solve_mma"
    return "k_pack_lower+k_cholesky_packed NT=128"


def rank_update_path(K):
    NB = kp(K) // 8
    if NB <= 13:
        return "launch_fused<%s>" % ("4,4,4" if NB <= 4 else "8,7,4" if NB <= 7 else "24,13,4")
    return "launch_pb_mma<%s>" % ("28,20,8" if NB <= 20 else "36,28,12")


# ---------------------------------------------------------------------------------------------------------------------
# extended-precision reference
# ---------------------------------------------------------------------------------------------------------------------
def sym_lower(M):
    """The symmetric matrix the lower triangle of M describes (what every device path reads)."""
    M = np.asarray(M)
    return np.tril(M) + np.swapaxes(np.tril(M, -1), -1, -2)


def chol_ld(M):
    """Batched Cholesky (n, K, K) -> L in longdouble: column by column, vectorised row updates."""
    A = sym_lower(np.asarray(M, dtype=LD)).copy()
    K = A.shape[-1]
    L = np.zeros_like(A)
    for j in range(K):
        d = np.sqrt(A[:, j, j])
        L[:, j, j] = d
        col = A[:, j + 1:, j] / d[:, None]
        L[:, j + 1:, j] = col
        A[:, j + 1:, j + 1:] -= col[:, :, None] * col[:, None, :]
    return L


def forward_ld(L, b):
    """y = L^-1 b."""
    y = np.array(b, dtype=LD)
    for j in range(L.shape[-1]):
        y[:, j] /= L[:, j, j]
        y[:, j + 1:] -= L[:, j + 1:, j] * y[:, j:j + 1]
    return y


def backward_ld(L, y):
    """x = L^-T y."""
    x = np.array(y, dtype=LD)
    for j in range(L.shape[-1] - 1, -1, -1):
        x[:, j] /= L[:, j, j]
        x[:, :j] -= L[:, j, :j] * x[:, j:j + 1]
    return x


def lt_times(L, d):
    """L^T d (batched)."""
    return (np.asarray(L, dtype=LD) * np.asarray(d, dtype=LD)[:, :, None]).sum(axis=1)


def quad_ld(L, d):
    """|L^T d|^2."""
    v = lt_times(L, d)
    return (v * v).sum(axis=1)


def kappa_eq(M):
    """2-norm condition number of the equilibrated matrix diag(M)^-1/2 M diag(M)^-1/2. Cholesky's rounding errors are
    componentwise relative to sqrt(M_ii M_jj), so this, not kappa(M), bounds the error of L relative to its row scale; for
    the well-scaled posterior matrices the two agree. (A tolerance needs kappa to a digit: float64 is plenty.)"""
    M = sym_lower(np.asarray(M, dtype=np.float64))
    s = 1.0 / np.sqrt(np.abs(np.diagonal(M, axis1=-2, axis2=-1)))
    w = np.linalg.eigvalsh(M * s[..., :, None] * s[..., None, :])
    return w[..., -1] / w[..., 0]


def tol_factor(K, kappa):
    """Relative tolerance of a factorisation-derived quantity: Cholesky's backward error is (K + 1) u |L||L^T|
    (Higham, Thm 10.3), the solution moves by the condition number times that; 4: slack for the solves on top."""
    return 4.0 * K * U * np.asarray(kappa, dtype=np.float64)


def assert_scaled(got, ref, weight, bound, what):
    """|got - ref| * weight <= bound for every matrix c (bound: per matrix). The message names the matrix, the element and
    its 8 x 8 block, which is what a broken block update or pivot shows up as."""
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - np.asarray(ref, dtype=LD)) * np.asarray(weight, dtype=LD)
    bound = np.broadcast_to(np.asarray(bound, dtype=np.float64), (len(err),))
    for c in range(len(err)):
        e = err[c]
        ok = e <= bound[c]            # NaN fails
        if not ok.all():
            idx = np.unravel_index(np.argmax(np.where(ok, -1.0, np.where(np.isnan(e), np.inf, e))), e.shape)
            raise AssertionError("%s: matrix %d, element %s (8x8 block %s): |error| %.3g > %.3g (got %r)" % (
                what, c, tuple(int(i) for i in idx), tuple(int(i) // 8 for i in idx), float(e[idx]), bound[c],
                float(got[c][idx])))


def row_scale(M):
    return np.sqrt(np.abs(np.diagonal(np.asarray(M, dtype=np.float64), axis1=-2, axis2=-1)))


def check_L(Ld, Lr, M, what):
    """L against the reference, element (i, j) relative to sqrt(M_ii) (|L_ij| <= sqrt(M_ii))."""
    K = Lr.shape[-1]
    assert_scaled(np.tril(Ld), np.tril(Lr), 1.0 / row_scale(M)[:, :, None], tol_factor(K, kappa_eq(M)), what)


def check_mu(mud, mur, M, what):
    """mu = D^-1 H^-1 D^-1 b (D = diag(M)^1/2, H equilibrated): D mu is what the condition number bounds."""
    r = row_scale(M)
    scale = np.abs(np.asarray(mur, dtype=np.float64) * r).max(axis=1)
    assert_scaled(mud, mur, r, tol_factor(M.shape[-1], kappa_eq(M)) * scale, what)


def check_y(yd, yr, M, what):
    """y = L^-1 b relative to max|y|."""
    scale = np.abs(np.asarray(yr, dtype=np.float64)).max(axis=1)
    assert_scaled(yd, yr, 1.0, tol_factor(M.shape[-1], kappa_eq(M)) * scale, what)


def check_q(qd, qr, scale, M, what):
    """|L^T w - y|^2: both terms carry the relative error above, the square doubles it; scale = (|L^T w| + |y|)^2."""
    assert_scaled(np.asarray(qd)[:, None], np.asarray(qr)[:, None], 1.0, 2.0 * tol_factor(M.shape[-1], kappa_eq(M)) * scale, what)


def backward_error(Ld, M):
    """max |L L^T - M| over the matrix, formed in longdouble, relative to max_i M_ii."""
    L = np.tril(np.asarray(Ld, dtype=LD))
    R = np.matmul(L, np.swapaxes(L, -1, -2)) - sym_lower(np.asarray(M, dtype=LD))
    return (np.abs(R).max(axis=(1, 2)) / np.abs(np.diagonal(M, axis1=-2, axis2=-1)).max(axis=1)).astype(np.float64)


# ---------------------------------------------------------------------------------------------------------------------
# data
# ---------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def twin(K, n=600):
    """Femur-like GPMM of rank K on an n-vertex mesh (Nystrom on 2K <= 448 points) and a model-instance target."""
    m = synth.femur_twin(rank=K, n=n)
    tv, tc, _ = synth.synthetic_target(m)
    m["target"], m["target_cells"] = tv, tc
    return m


@functools.lru_cache(maxsize=None)
def oracle_pair(K, n=600):
    m = twin(K, n)
    return orc.Model(m["ref"], m["cells"], m["basis"], m["variance"]), orc.Mesh(m["target"], m["target_cells"])


def obs_lists(m, K, n_obs=None):
    """n_obs model point ids and target points (default 2K, at least 24); drawn with repetition beyond the mesh size."""
    n_obs = n_obs or max(2 * K, 24)
    rng = np.random.default_rng(K * 1009 + n_obs)
    N, tv = len(m["ref"]), m["target"]
    ids = np.sort(rng.choice(N, n_obs, replace=n_obs > N))
    tp = tv[np.sort(rng.choice(len(tv), n_obs, replace=n_obs > len(tv)))] + rng.normal(0, 0.2, (n_obs, 3))
    return ids, tp


@functools.lru_cache(maxsize=None)
def factor_data(K):
    """Five matrices at rank K with right-hand sides, transition thetas and their longdouble factorisation: I + A^T A with
    2K and 3K rows (scaled to the diagonal of the femur-like posterior), graded D (I + A^T A) D with kappa(M) ~ 1e8 and 1e12,
    and the oracle's own posterior matrix. The graded pair keeps the equilibrated condition number of I + A^T A, which is what
    the tolerances use: they check that the factorisation does not lose accuracy to the diagonal scaling."""
    m = twin(K)
    ids, tp = obs_lists(m, K)
    om, ot = oracle_pair(K)
    op = orc.IcpProposal(om, ot, STEP, 10.0, 5.0, orc.MODEL_SAMPLING, True, ids, tp)
    rng = np.random.default_rng(100 + K)
    po = op.posterior(random_theta(m, rng, 1)[0])
    Mo = po["M"]
    scale = Mo.diagonal().max()
    mats, names = [], []
    for rows in (2, 3):
        A = rng.normal(size=(rows * K, K)) * np.sqrt(scale / (rows * K))
        mats.append(np.eye(K) + A.T @ A)
        names.append("I+AtA(%dK rows)" % rows)
    for target in (1e8, 1e12):
        # D = diag(10^-e t), t in [0, 1]: kappa(M) grows with e about as 10^2e; one correction of e lands near the target
        e, G = 0.0, mats[0]
        for _ in range(3 if K > 1 else 0):
            e += 0.5 * np.log10(target / np.linalg.cond(G))
            g = 10.0 ** (-e * np.linspace(0.0, 1.0, K))
            G = g[:, None] * mats[0] * g[None, :]
        mats.append(G)
        names.append("graded(kappa(M)=%.1e)" % np.linalg.cond(G))
    mats.append(Mo)
    names.append("oracle posterior")
    M = sym_lower(np.stack(mats))
    nd = len(M)
    b = rng.normal(size=(nd, K)) * row_scale(M)
    b[-1] = (Mo.astype(LD) @ po["mu"].astype(LD)).astype(np.float64)
    th = np.zeros((nd, K + 10))
    th[:, 0] = 1.0
    th[:, 10:] = rng.normal(0, 0.3, (nd, K))
    to = th.copy()
    to[:, 10:] += STEP * rng.normal(0, 0.3, (nd, K))
    w = th[:, 10:] + (to[:, 10:] - th[:, 10:]) / STEP        # the device's float64 arithmetic for the transition point
    Lr = chol_ld(M)
    yr = forward_ld(Lr, b)
    mur = backward_ld(Lr, yr)
    qr = quad_ld(Lr, w - mur)
    qscale = (np.sqrt((lt_times(Lr, w) ** 2).sum(1)) + np.sqrt((yr * yr).sum(1))).astype(np.float64) ** 2
    return dict(names=names, M=M, b=b, th=th, to=to, L=Lr, y=yr, mu=mur, q=qr, qscale=qscale)


def factor(ctx, M, b, th=None, to=None, ymean=False):
    """icp_debug_factor with L pre-filled with SENTINEL (the entry writes the lower triangle only)."""
    M = np.ascontiguousarray(M, dtype=np.float64)
    c, K = M.shape[0], M.shape[1]
    b = np.ascontiguousarray(b, dtype=np.float64).reshape(c, K)
    L = np.full((c, K, K), SENTINEL)
    mean = np.empty((c, K))
    st = np.full(c, -1, np.int32)
    q = tp = tq = None
    if th is not None:
        q = np.empty(c)
        tp = np.ascontiguousarray(th, dtype=np.float64)
        tq = np.ascontiguousarray(to, dtype=np.float64)
    _lib.check(ctx.lib.icp_debug_factor(ctx.h, c, K, _lib.dptr(M), _lib.dptr(b), None if tp is None else _lib.dptr(tp),
                                        None if tq is None else _lib.dptr(tq), float(STEP), int(bool(ymean)), _lib.dptr(L),
                                        _lib.dptr(mean), None if q is None else _lib.dptr(q), _lib.iptr(st)), ctx.h)
    return L, mean, q, st


# ---------------------------------------------------------------------------------------------------------------------
# (a) the factorisation alone
# ---------------------------------------------------------------------------------------------------------------------
def batch_sizes(K):
    # Kp <= 104: C <= 148 runs NT = 256, C > 148 NT = 128; above, one form only
    return (1, 148, 149, 333) if kp(K) <= 104 else (1, 149)


def check_factor(ctx, K, Cs=None):
    """The factorisation at rank K against the longdouble reference, and its bit-for-bit invariances."""
    d = factor_data(K)
    M, b, th, to = d["M"], d["b"], d["th"], d["to"]
    nd = len(M)
    iu = np.triu_indices(K, 1)
    single = {}
    for ymean in (False, True):
        runs = [factor(ctx, M[i:i + 1], b[i:i + 1], th[i:i + 1], to[i:i + 1], ymean) for i in range(nd)]
        L, mean, q, st = (np.concatenate([r[k] for r in runs]) for k in range(4))
        single[ymean] = (L, mean, q, st)
        form = "y form" if ymean else "mu form"
        for i in range(nd):
            what = "K=%d %s, %s, %s" % (K, factor_path(K, 1), form, d["names"][i])
            assert st[i] == 0, what + ": status %d" % st[i]
            assert (L[i][iu] == SENTINEL).all(), what + ": the upper triangle of L was written"
            be = backward_error(L[i:i + 1], M[i:i + 1])[0]
            assert be <= 4.0 * K * U, what + ": backward error %.3g > 4 K u = %.3g" % (be, 4.0 * K * U)
            check_L(L[i:i + 1], d["L"][i:i + 1], M[i:i + 1], what + ": L")
            if ymean:
                check_y(mean[i:i + 1], d["y"][i:i + 1], M[i:i + 1], what + ": y = L^-1 b")
            else:
                check_mu(mean[i:i + 1], d["mu"][i:i + 1], M[i:i + 1], what + ": mu")
            check_q(q[i:i + 1], d["q"][i:i + 1], d["qscale"][i:i + 1], M[i:i + 1], what + ": q")
    assert np.array_equal(single[False][0], single[True][0]), "K=%d: L differs between the mu and the y form" % K
    for C in Cs or batch_sizes(K):
        idx = np.arange(C) % nd      # every slot holds one of the five matrices: each must reproduce its C = 1 run
        for ymean in (False, True):
            got = factor(ctx, M[idx], b[idx], th[idx], to[idx], ymean)
            for k, name in enumerate(("L", "mean", "q", "status")):
                want = single[ymean][k][idx]
                same = np.array([np.array_equal(got[k][c], want[c]) for c in range(C)])
                assert same.all(), "K=%d C=%d (%s) vs C=1 (%s), %s form: %s of slot %d differs" % (
                    K, C, factor_path(K, C), factor_path(K, 1), "y" if ymean else "mu", name, int(np.argmin(same)))
    # NaN in the strictly upper triangle of M changes nothing: every path reads the lower triangle only
    C = max(Cs or batch_sizes(K))
    idx = np.arange(C) % nd
    Mn = M[idx].copy()
    Mn[:, iu[0], iu[1]] = np.nan
    for ymean in (False, True):
        got = factor(ctx, Mn, b[idx], th[idx], to[idx], ymean)
        for k, name in enumerate(("L", "mean", "q", "status")):
            assert np.array_equal(got[k], single[ymean][k][idx]), "K=%d C=%d (%s): NaN above the diagonal of M changed %s" % (
                K, C, factor_path(K, C), name)


@pytest.mark.parametrize("K", RANKS, ids=["K%d-%s" % (K, factor_path(K, 149).split()[0]) for K in RANKS])
def test_factorisation_against_extended_reference(ctx, K):
    """Backward error, L, mu, y and q against the longdouble reference on five matrix families; the same bits at every
    batch position and size (NT = 256 vs NT = 128 of k_cholesky_packed for Kp <= 104), in both forms, with NaN above the
    diagonal; the upper triangle of L untouched. Paths: k_cholesky_packed (Kp <= 104), k_cholesky_solve_mma
    (104 < Kp <= 160), k_pack_lower + k_cholesky_packed (160 < Kp <= 224, near-full shared memory at Kp = 224)."""
    check_factor(ctx, K)


# ---------------------------------------------------------------------------------------------------------------------
# (b) failure isolation
# ---------------------------------------------------------------------------------------------------------------------
def _break(M, L, case):
    K = len(M)
    M = M.copy()
    if case.startswith("negative_pivot"):
        r = {"negative_pivot_row0": 0, "negative_pivot_block_end": 8 * ((K // 8) // 2) + 7, "negative_pivot_last": K - 1}[case]
        M[r, r] = float((L[r, :r].astype(LD) ** 2).sum()) - 1.0      # Schur pivot -1 (M_ii ~ 1e3: far from rounding)
    elif case == "zero_pivot":
        r = K // 2
        M[r, :] = 0.0
        M[:, r] = 0.0                                                  # decoupled row: the pivot is exactly 0
    elif case == "nan_diagonal":
        M[K // 3, K // 3] = np.nan
    elif case == "inf_diagonal_last":
        M[K - 1, K - 1] = np.inf                                       # the last pivot: nothing after it turns it into NaN
    elif case == "inf_diagonal_row0":
        M[0, 0] = np.inf
    return M


FAIL_CASES = ("negative_pivot_row0", "negative_pivot_block_end", "negative_pivot_last", "zero_pivot", "nan_diagonal",
              "inf_diagonal_last", "inf_diagonal_row0")


def check_failure_isolation(ctx, K, C):
    """One matrix that is not positive definite among good ones: status 1 and NaN in its L and mean; every other matrix
    bit-identical to a run without it."""
    d = factor_data(K)
    nd = len(d["M"])
    idx = np.arange(C) % nd
    M, b = d["M"][idx], d["b"][idx]
    L0, m0, _, s0 = factor(ctx, M, b)
    assert (s0 == 0).all()
    tri = np.tril_indices(K)
    for case in FAIL_CASES:
        p = C - 1 if case.endswith("last") else C // 2
        Mb = M.copy()
        Mb[p] = _break(M[p], d["L"][idx[p]], case)
        L, mean, _, st = factor(ctx, Mb, b)
        what = "K=%d C=%d (%s) %s at slot %d" % (K, C, factor_path(K, C), case, p)
        assert st[p] == 1, what + ": status %d" % st[p]
        assert np.isnan(L[p][tri]).all() and np.isnan(mean[p]).all(), what + ": L / mean not NaN"
        others = np.arange(C) != p
        assert (st[others] == 0).all(), what
        assert np.array_equal(L[others], L0[others]) and np.array_equal(mean[others], m0[others]), what + ": other matrices changed"


@pytest.mark.parametrize("C", [5, 149])
@pytest.mark.parametrize("K", [40, 120, 224], ids=["K40-k_cholesky_packed", "K120-k_cholesky_solve_mma",
                                                    "K224-k_pack_lower+k_cholesky_packed"])
def test_failure_isolation(ctx, K, C):
    """Negative pivots at row 0, at the last row of an 8-row block and at row K - 1, an exact zero pivot, NaN and +Inf on the
    diagonal (+Inf at row K - 1 used to leave status 0 with NaN in L: rsqrt(Inf) = 0 turns into NaN only after the test)."""
    check_failure_isolation(ctx, K, C)


# ---------------------------------------------------------------------------------------------------------------------
# (c) the posterior pipeline
# ---------------------------------------------------------------------------------------------------------------------
def run_proposal(gp, th, z):
    mu, M, n = gp.posterior(th)
    prop = gp.propose(th, z)
    return dict(mu=mu, M=M, n=n, prop=prop, lt=gp.log_transition(th, prop), ltb=gp.log_transition(prop, th))


def assert_same(a, b, what):
    for k in a:
        assert np.array_equal(a[k], b[k]), "%s: %s differs" % (what, k)


def check_pipeline(ctx, K, mode, C=149, n_model=600, n_obs=None, check=(0, -1), rank_update=_lib.RANK_UPDATE_FP64):
    """icp_posterior / icp_propose / icp_log_transition at rank K against the oracle's closed forms on the chains in
    `check`, and every chain of a C = 1 run of those chains bit-identical to its slot in the batch."""
    m = twin(K, n_model)
    ids, tp = obs_lists(m, K, n_obs)
    direction, sd_t, sd_n = MODES[mode]
    om, ot = oracle_pair(K, n_model)
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    gp = core.IcpProposal(model, tgt, STEP, sd_t, sd_n, direction, True, ids, tp, rank_update=rank_update)
    op = orc.IcpProposal(om, ot, STEP, sd_t, sd_n, direction, True, ids, tp)
    tag = "K=%d (%s) %s n_obs=%d C=%d" % (K, rank_update_path(K), mode, len(ids), C)
    try:
        rng = np.random.default_rng(K * 7 + len(ids))
        th = random_theta(m, rng, C, alpha_sd=0.3)
        z = rng.normal(size=(C, K))
        got = run_proposal(gp, th, z)
        assert np.array_equal(got["prop"][:, :10], th[:, :10]), tag + ": the pose part of a proposal changed"
        # the twin is closed: every observation is kept, which model_rpo1 needs to stay on the constant-Gram path (all_kept)
        assert (got["n"] == len(ids)).all(), tag + ": observations dropped"
        for c in sorted({x % C for x in check}):
            po = op.posterior(th[c])
            what = "%s chain %d" % (tag, c)
            assert got["n"][c] == po["n"], what
            Mo = po["M"]
            rows = 3 * int(po["n"]) + K          # products summed into an element of M (and b)
            # M: a sum of `rows` products, each within a few u of the oracle's: (rows) u relative to max|M|, 4 for slack
            # (the INT8 emulation: its own accuracy)
            m_tol = I8_BOUND if rank_update == _lib.RANK_UPDATE_INT8 else 4.0 * rows * U
            dM = np.abs(got["M"][c] - Mo).max() / np.abs(Mo).max()
            assert dM <= m_tol, what + ": M off by %.3g relative > %.3g" % (dM, m_tol)
            # the solution moves by kappa times the relative difference of the inputs (measured on M, the bound on b)
            t = 4.0 * kappa_eq(Mo[None])[0] * (dM + rows * U)
            r = row_scale(Mo[None])[0]
            assert_scaled(got["mu"][c:c + 1], po["mu"][None], r, t * np.abs(po["mu"] * r).max(), what + ": mu")
            want = op.propose(th[c], z[c], closed_form=True)
            assert_scaled(got["prop"][c:c + 1, 10:], want[None, 10:], 1.0, t * (np.abs(want[10:]).max() + np.abs(th[c, 10:]).max()),
                          what + ": proposal")
            for key, f, to_ in (("lt", th[c], got["prop"][c]), ("ltb", got["prop"][c], th[c])):
                w = op.log_transition(f, to_, closed_form=True)
                assert_scaled(got[key][c:c + 1, None], np.array([[w]]), 1.0, t * (abs(w) + K), what + ": " + key)
        if C > 1:
            for c in (0, C - 1):
                gp.clear_cache()        # the C = 1 run forms its own posterior instead of finding the batch's in the cache
                one = run_proposal(gp, th[c:c + 1], z[c:c + 1])
                assert_same(one, {k: v[c:c + 1] for k, v in got.items()}, "%s: C = 1 run of chain %d" % (tag, c))
        return got, th, z
    finally:
        gp.close(); model.close(); tgt.close()


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("K", RANKS, ids=["K%d-%s" % (K, rank_update_path(K)) for K in RANKS])
def test_posterior_pipeline(ctx, K, mode):
    """M, mu, the proposal for a fixed z and both transition densities against the oracle, C = 149 with chains 0 and 148
    also run alone (bit for bit). model_rpo1: the constant-Gram rank update (one row per observation), model_rpo3 and
    target: the general three-row update. Rank updates: launch_fused<4,4,4> / <8,7,4> / <24,13,4> (NB <= 13) and
    launch_pb_mma<28,20,8> / <36,28,12> (NB 14..28) at the first and last rank of every bucket."""
    check_pipeline(ctx, K, mode)


@pytest.mark.parametrize("mode", ["model_rpo1", "model_rpo3", "target"])
@pytest.mark.parametrize("n_obs", [4096, 4097])
@pytest.mark.parametrize("K", [57, 105, 224], ids=["K57-k_posterior_fused", "K105-k_posterior_build_mma",
                                                   "K224-k_posterior_build_mma"])
def test_observation_staging(ctx, K, n_obs, mode):
    """kMaxStagedIds = 4096: 4096 observations stage their vertex ids in shared memory, 4097 take the unstaged branch of
    the rank update (6000-vertex model)."""
    check_pipeline(ctx, K, mode, C=4, n_model=6000, n_obs=n_obs)


@pytest.mark.parametrize("mode", ["model_rpo1", "model_rpo3"])
@pytest.mark.parametrize("K", [105, 112])
def test_int8_rank_update_at_widest_tile(ctx, K, mode):
    """Kp = 112, the widest INT8 tile: against the FP64 path of the library on every chain. With C = 149 on 148 SMs chain
    148 is the second chain of its persistent CTA (its first step converted during chain 0's epilogue): the C = 1 run of it
    must give the same bits (b used to sum in a different order there)."""
    got, th, z = check_pipeline(ctx, K, mode, C=149, rank_update=_lib.RANK_UPDATE_INT8)
    m = twin(K)
    ids, tp = obs_lists(m, K)
    direction, sd_t, sd_n = MODES[mode]
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    gf = core.IcpProposal(model, tgt, STEP, sd_t, sd_n, direction, True, ids, tp)
    ref = run_proposal(gf, th, z)
    gf.close(); model.close(); tgt.close()
    err = np.abs(got["M"] - ref["M"]).max(axis=(1, 2)) / np.abs(ref["M"]).max(axis=(1, 2))
    assert err.max() <= I8_BOUND and err.max() > 0.0, err.max()       # > 0: the INT8 kernel ran, not the FP64 one
    kap = kappa_eq(ref["M"])
    r = row_scale(ref["M"])
    assert_scaled(got["mu"], ref["mu"], r, 4.0 * kap * I8_BOUND * np.abs(ref["mu"] * r).max(axis=1), "K=%d %s INT8 mu" % (K, mode))


@pytest.mark.parametrize("K,n_obs,mode", [(113, None, "model_rpo1"), (113, None, "model_rpo3"), (105, 10667, "model_rpo3")],
                         ids=["Kp120-rpo1", "Kp120-rpo3", "Kp112-10667obs-rpo3"])
def test_int8_fallback_is_the_fp64_path(ctx, K, n_obs, mode):
    """Outside the INT8 kernel's domain (Kp > 112, or n * rows per observation > 32000; tc_i8.cu) rank_update=INT8 runs
    the FP64 path: bit-identical results, where a wrong kernel would differ in the last bits at least."""
    m = twin(K)
    ids, tp = obs_lists(m, K, n_obs)
    direction, sd_t, sd_n = MODES[mode]
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    rng = np.random.default_rng(K)
    th = random_theta(m, rng, 7, alpha_sd=0.3)
    z = rng.normal(size=(7, K))
    out = []
    for ru in (_lib.RANK_UPDATE_INT8, _lib.RANK_UPDATE_FP64):
        gp = core.IcpProposal(model, tgt, STEP, sd_t, sd_n, direction, True, ids, tp, rank_update=ru)
        out.append(run_proposal(gp, th, z))
        gp.close()
    model.close(); tgt.close()
    assert (out[1]["n"] == len(ids)).all()
    assert_same(out[0], out[1], "K=%d n_obs=%d %s: INT8 fallback vs FP64" % (K, len(ids), mode))


# ---------------------------------------------------------------------------------------------------------------------
# (d) the SVD factor
# ---------------------------------------------------------------------------------------------------------------------
def svd_branch(K):
    return "HJ-shared" if kp(K) <= 112 else "one-global" if kp(K) <= 160 else "both-global"


@pytest.mark.parametrize("K", [105, 113, 160, 161, 201, 224], ids=lambda K: "K%d-%s" % (K, svd_branch(K)))
def test_svd_factor(ctx, K):
    """factor=FACTOR_SVD in each shared-memory branch of launch_svd_factor: the proposal against the oracle's reference
    structure, W W^T = M^-1 against the longdouble inverse, W^T M W = I (the columns the Jacobi sweeps orthogonalise), and
    the sweep count of the Jacobi loop (icp_debug_svd_factor) below its cap of 40."""
    m = twin(K)
    ids, tp = obs_lists(m, K)
    om, ot = oracle_pair(K)
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    step = 1.0       # alpha' = S v: the columns of S W are read off without cancellation
    gs = core.IcpProposal(model, tgt, step, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp, factor=_lib.FACTOR_SVD)
    gc = core.IcpProposal(model, tgt, step, 10.0, 5.0, _lib.MODEL_SAMPLING, True, ids, tp)
    op = orc.IcpProposal(om, ot, step, 10.0, 5.0, orc.MODEL_SAMPLING, True, ids, tp)
    rng = np.random.default_rng(K + 5)
    th = random_theta(m, rng, 1, alpha_sd=0.3)
    z = rng.normal(size=(1, K))
    try:
        _, M, _ = gs.posterior(th)
        kap = kappa_eq(M)[0]
        # eigenvectors of Sigma' = D M^-1 D are determined to u kappa / (relative eigenvalue gap)
        D = np.sqrt(m["variance"])
        lam = np.linalg.eigvalsh(D[:, None] * np.linalg.inv(M[0]) * D[None, :])
        gap = max(np.diff(lam).min() / lam[-1], U)
        # the reference structure maps the sample back to coefficients through the eps = 1e-5 regularised regression on the
        # whole mesh, (Q^T Q / eps + I) a = Q^T d / eps, solved in float64: its condition number enters as well
        Q = m["basis"] * np.sqrt(m["variance"])
        kap_reg = np.linalg.cond(Q.T @ Q / 1e-5 + np.eye(K))
        prop = gs.propose(th, z)[0]
        want = op.propose(th[0], z[0])
        tol = 4.0 * U * (K * kap / gap + kap_reg)
        assert_scaled(prop[None, 10:], want[None, 10:], 1.0, tol * np.abs(want[10:]).max(), "K=%d SVD proposal" % K)
        # P = S W from propose with z = e_i (minus z = 0); the Cholesky proposal gives S L^-T, so S = P_chol L^T
        thK = np.repeat(th, K, axis=0)
        P = (gs.propose(thK, np.eye(K))[:, 10:] - gs.propose(th, np.zeros((1, K)))[0, 10:]).T
        Pc = (gc.propose(thK, np.eye(K))[:, 10:] - gc.propose(th, np.zeros((1, K)))[0, 10:]).T
        Lr = chol_ld(M)[0]
        S = Pc.astype(LD) @ Lr.T
        Lb = np.broadcast_to(Lr, (K, K, K))
        Minv = backward_ld(Lb, forward_ld(Lb, np.eye(K)))     # row i: M^-1 e_i
        cov = S @ Minv @ S.T
        t = tol_factor(K, kap)
        assert_scaled((P.astype(LD) @ P.T.astype(LD))[None].astype(np.float64), cov[None], 1.0, t * float(np.abs(cov).max()),
                      "K=%d (%s): W W^T vs M^-1" % (K, svd_branch(K)))
        W = np.linalg.solve(S.astype(np.float64), P)
        G = W.T.astype(LD) @ sym_lower(M[0].astype(LD)) @ W.astype(LD)
        assert_scaled(G[None].astype(np.float64), np.eye(K)[None], 1.0, t, "K=%d (%s): W^T M W vs I" % (K, svd_branch(K)))
        # the factor alone, from the device's Cholesky factor of the same M: the Jacobi loop must stop on its own, inside
        # kSvdMaxSweeps = 40 (a loop that ran into the cap would still leave W W^T = M^-1 to rounding, so the checks above
        # cannot tell), and its W must be the one the proposal samples with
        Ld = np.tril(factor(ctx, M, np.zeros((1, K)))[0])
        Wd, sweeps = ctx.svd_factor(Ld, m["variance"])
        assert sweeps[0] < 40, "K=%d (%s): the Jacobi sweeps ran into their cap" % (K, svd_branch(K))
        assert_scaled((Wd[0].astype(LD) @ Wd[0].T.astype(LD))[None].astype(np.float64), Minv[None], 1.0,
                      t * float(np.abs(Minv).max()), "K=%d (%s): W W^T vs M^-1 (icp_debug_svd_factor)" % (K, svd_branch(K)))
        assert_scaled(P[None], (S @ Wd[0].astype(LD))[None], 1.0, t * float(np.abs(P).max()),
                      "K=%d (%s): the proposal's factor vs icp_debug_svd_factor" % (K, svd_branch(K)))
    finally:
        gs.close(); gc.close(); model.close(); tgt.close()


# ---------------------------------------------------------------------------------------------------------------------
# (e) the device-resident runners
# ---------------------------------------------------------------------------------------------------------------------
EDGE_RANKS = (1, 9, 105, 161, 224)
STD_ICP_RANKS = (1, 9, 56, 57, 104, 105, 161, 224)     # both ends of the k_si_project<7> and <13> buckets, and <28>


@pytest.mark.parametrize("K", EDGE_RANKS)
def test_chain_at_edge_ranks(ctx, K):
    """20 fused MH steps (ICP target and model sampling + random walk, caller-supplied randomness) against the oracle chain.
    At K = 224 k_chain_propose holds the packed factor in 214 KB of shared memory."""
    m = twin(K)
    ids, tp = obs_lists(m, K)
    om, ot = oracle_pair(K)
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    mk = lambda d: core.IcpProposal(model, tgt, STEP, 10.0, 5.0, d, True, ids, tp)
    mo = lambda d: orc.IcpProposal(om, ot, STEP, 10.0, 5.0, d, True, ids, tp)
    comps = [dict(kind=0, weight=0.45, proposal=mk(1)), dict(kind=0, weight=0.45, proposal=mk(0)), dict(kind=1, weight=0.1, sd=0.1)]
    comps_o = [dict(kind=0, weight=0.45, icp=mo(1)), dict(kind=0, weight=0.45, icp=mo(0)), dict(kind=1, weight=0.1, sd=0.1)]
    ev = core.Evaluator(model, tgt, _lib.EVAL_INDEPENDENT, 0, True, 0.0, 2.0, 0.0, ids, tp)
    chain = core.Chain(model, tgt, comps, ev, max_chains=2)
    rng = np.random.default_rng(300 + K)
    n, C = 20, 2
    th0 = random_theta(m, rng, C, alpha_sd=0.5)
    u_comp, u_acc, z = rng.random((n, C)), rng.random((n, C)), rng.normal(size=(n, C, K))
    got = chain.run(th0, n, u_comp=u_comp, z=z, u_acc=u_acc)
    # every step adds the rounding of one posterior solve: n steps of 4 kappa (3 n_obs + K) u
    kap = kappa_eq(factor_data(K)["M"][-1:])[0]
    t = n * 4.0 * kap * (3 * len(ids) + K) * U
    try:
        assert np.all(got["status"] == 0)
        for c in range(C):
            want = orc.chain_run(om, ot, comps_o, True, orc.EVAL_INDEPENDENT, 0, (0.0, 2.0), ids, tp, th0[c], n, u_comp[:, c],
                                 z[:, c], u_acc[:, c], closed_form=True)
            what = "K=%d chain %d" % (K, c)
            assert np.array_equal(got["component"][:, c], want["comp"]), what
            assert np.array_equal(got["accepted"][:, c], want["accepted"]), what
            assert_scaled(got["values"][None, :, c], want["logv"][None], 1.0, t * np.abs(want["logv"]).max(), what + ": values")
            assert_scaled(got["theta"][None, :, c], want["theta"][None], 1.0, t * np.abs(want["theta"]).max(), what + ": theta")
    finally:
        chain.close(); ev.close()
        for cp in comps[:2]:
            cp["proposal"].close()
        model.close(); tgt.close()


@pytest.mark.parametrize("K", STD_ICP_RANKS, ids=lambda K: "K%d-k_si_project<%d>" % (K, 7 if kp(K) <= 56 else 13 if kp(K) <= 104 else 28))
def test_std_icp_at_edge_ranks(ctx, K):
    """A 5-iteration StdIcp run (fit 0 model sampling, fit 1 target sampling) against the per-call iteration row by row."""
    m = twin(K)
    ids, tp = obs_lists(m, K)
    model, tgt = core.Model(ctx, m["ref"], m["cells"], m["basis"], m["variance"]), core.Target(ctx, m["target"], m["target_cells"])
    runner = core.StdIcp(model, tgt, ids, tp, 1.0, _lib.MODEL_SAMPLING, max_fits=2)
    rng = np.random.default_rng(400 + K)
    th0 = random_theta(m, rng, 2, alpha_sd=0.3)
    th0[:, 7:10] = 0.0
    sigma2, n_it = (1.0,), 4
    iters = n_it + 1
    dirs = np.tile(np.array([[0, 1]], np.int32), (iters, 1))
    try:
        out = runner.run(th0, sigma2, n_it, directions=dirs)
        assert (out["status"] == 0).all() and (out["iterations_done"] == iters).all()
        want = np.empty_like(out["log_alpha"])
        for it in range(iters):
            prev = th0[:, 10:] if it == 0 else out["log_alpha"][it - 1]
            for dd in (0, 1):
                want[it, dd:dd + 1] = core.std_icp_iteration(model, tgt, dd, ids, tp, sigma2[0], 1.0, prev[dd:dd + 1])
        # kappa(I + Q^T Q / sigma^2) <= 1 + n_obs max_v |Q_v|_F^2 / sigma^2 (every observation adds at most |Q_v|^2)
        Q = m["basis"] * np.sqrt(m["variance"])
        kap = 1.0 + len(ids) * (Q.reshape(-1, 3, K) ** 2).sum(axis=(1, 2)).max() / sigma2[0]
        t = 4.0 * kap * (3 * len(ids) + K) * U
        assert_scaled(out["log_alpha"].reshape(1, -1), want.reshape(1, -1), 1.0, t * np.abs(want).max(), "K=%d StdIcp" % K)
    finally:
        runner.close(); model.close(); tgt.close()


# ---------------------------------------------------------------------------------------------------------------------
# (f) environment-selected paths, and the rank limit
# ---------------------------------------------------------------------------------------------------------------------
CHILD_RANKS = (33, 104, 113, 161)


@pytest.mark.parametrize("var", ["ICPCUDA_NO_DMMA", "ICPCUDA_FUSE"])
def test_environment_selected_paths(var):
    """ICPCUDA_NO_DMMA=1: k_posterior_build + k_cholesky_solve (+ k_mean_to_ymean); ICPCUDA_FUSE=1: the single-launch
    k_posterior_fused<.., true>. Read once per process, so a child process runs the checks of (a), (b) and (c) and reports
    (k_cholesky_solve, at K = 113, used to let +Inf on the diagonal through: 1 / sqrt(Inf) zeroes the column)."""
    env = dict(os.environ, **{var: "1"})
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), "--child"]
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=1800, cwd=os.path.dirname(os.path.abspath(__file__)))
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("CHILD-SUMMARY ")]
    assert r.returncode == 0 and lines, (r.returncode, r.stdout[-2000:], r.stderr[-4000:])
    res = json.loads(lines[-1][len("CHILD-SUMMARY "):])
    assert len(res) == len(CHILD_RANKS) * (2 + len(MODES)), res
    failed = {k: v for k, v in res.items() if v != "pass"}
    assert not failed, failed


def test_rank_above_224_is_refused(ctx):
    """icp_model_create and icp_debug_factor both take 1 <= K <= 224 (K = 225 would still fit the packed factorisation)."""
    L, _, _, st = factor(ctx, np.eye(224)[None], np.zeros((1, 224)))
    assert st[0] == 0 and np.array_equal(np.tril(L[0]), np.eye(224))
    with pytest.raises(_lib.IcpCudaError) as e:
        factor(ctx, np.eye(225)[None], np.zeros((1, 225)))
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT
    m = twin(8)
    basis = np.random.default_rng(0).normal(size=(3 * len(m["ref"]), 225))
    with pytest.raises(_lib.IcpCudaError) as e:
        core.Model(ctx, m["ref"], m["cells"], basis, np.ones(225))
    assert e.value.code == _lib.ERR_INVALID_ARGUMENT


def _child():
    ctx = core.Context(0)
    res = {}
    try:
        for K in CHILD_RANKS:
            checks = [("factor", lambda K=K: check_factor(ctx, K, (1, 149))),
                      ("failure", lambda K=K: check_failure_isolation(ctx, K, 5))]
            checks += [("pipeline-" + mode, lambda K=K, mode=mode: check_pipeline(ctx, K, mode)) for mode in MODES]
            for name, fn in checks:
                try:
                    fn()
                    res["K=%d %s" % (K, name)] = "pass"
                except Exception as e:       # report every check, not only the first failure
                    res["K=%d %s" % (K, name)] = "FAIL: %s" % e
    finally:
        ctx.close()
    print("CHILD-SUMMARY " + json.dumps(res), flush=True)


if __name__ == "__main__" and "--child" in sys.argv:
    _child()
