"""The longdouble reference and the tolerance helpers of tests/test_gpu_posterior_ranks.py, without a GPU: the reference
agrees with LAPACK to float64 rounding, and the helpers reject the errors a broken factorisation kernel makes. Without
these, a passing GPU comparison would say nothing."""
import numpy as np
import pytest
import scipy.linalg as sla

from test_gpu_posterior_ranks import (LD, U, backward_error, backward_ld, check_L, check_mu, check_q, check_y, chol_ld,
                                      forward_ld, kappa_eq, lt_times, quad_ld, tol_factor)


def _spd(K, rows, seed, n=3):
    rng = np.random.default_rng(seed)
    A = rng.normal(size=(n, rows, K)) * np.sqrt(1e3 / rows)
    M = np.eye(K) + np.einsum("cri,crj->cij", A, A)
    M = np.tril(M) + np.swapaxes(np.tril(M, -1), -1, -2)
    b = rng.normal(size=(n, K)) * 30.0
    return M, b


def _reference(M, b):
    L = chol_ld(M)
    y = forward_ld(L, b)
    return L, y, backward_ld(L, y)


def _blocked_cholesky(M, skip=None):
    """Right-looking 8 x 8 blocked Cholesky in float64; skip = (bi, bj, p): block (bi, bj) misses the update from block
    column p, the error a dropped DMMA update in the device kernels makes."""
    A = M.copy()
    K = len(A)
    NB = (K + 7) // 8
    blk = lambda i: slice(8 * i, min(8 * i + 8, K))
    for p in range(NB):
        A[blk(p), blk(p)] = np.linalg.cholesky(A[blk(p), blk(p)])
        below = slice(8 * p + 8, K)
        A[below, blk(p)] = sla.solve_triangular(A[blk(p), blk(p)], A[below, blk(p)].T, lower=True).T
        for bi in range(p + 1, NB):
            for bj in range(p + 1, bi + 1):
                if skip != (bi, bj, p):
                    A[blk(bi), blk(bj)] -= A[blk(bi), blk(p)] @ A[blk(bj), blk(p)].T
    return np.tril(A)


@pytest.mark.parametrize("K", [1, 9, 57, 113])
def test_reference_agrees_with_lapack(K):
    M, b = _spd(K, 2 * K + 3, K)
    L, y, mu = _reference(M, b)
    kap = kappa_eq(M)
    for c in range(len(M)):
        Lc = np.tril(sla.cho_factor(M[c], lower=True)[0])
        muc = sla.cho_solve((Lc, True), b[c])
        # LAPACK's own error is what separates the two: the Cholesky bound for float64 against a 1e-19 reference
        t = tol_factor(K, kap[c])
        r = np.sqrt(np.diag(M[c]))
        assert (np.abs(Lc - L[c].astype(float)) / r[:, None]).max() <= t
        assert (np.abs(muc - mu[c].astype(float)) * r).max() <= t * np.abs(mu[c].astype(float) * r).max()
        yc = sla.solve_triangular(Lc, b[c], lower=True)
        assert np.abs(yc - y[c].astype(float)).max() <= t * np.abs(yc).max()
    w = np.random.default_rng(1).normal(size=(len(M), K))
    q = quad_ld(L, w - mu)
    q64 = np.einsum("ci,cij,cj->c", w - mu.astype(float), M, w - mu.astype(float))
    np.testing.assert_allclose(q.astype(float), q64, rtol=8 * K * U * kap.max())
    # the reference itself: L L^T = M to longdouble rounding, far below the device tolerance
    assert backward_error(L, M).max() <= 4 * K * float(np.finfo(LD).eps)


def test_helpers_accept_float64_rounding_of_the_reference():
    M, b = _spd(32, 96, 3)
    L, y, mu = _reference(M, b)
    check_L(L.astype(float), L, M, "rounded reference")
    check_mu(mu.astype(float), mu, M, "rounded reference")
    check_y(y.astype(float), y, M, "rounded reference")
    w = np.random.default_rng(2).normal(size=(len(M), 32))
    q = quad_ld(L, w - mu)
    scale = (np.sqrt((lt_times(L, w) ** 2).sum(1)) + np.sqrt((y * y).sum(1))).astype(float) ** 2
    check_q(q.astype(float), q, scale, M, "rounded reference")


def test_rejects_one_element_off_by_1e_12():
    M, b = _spd(32, 96, 4)
    L, _, _ = _reference(M, b)
    assert tol_factor(32, kappa_eq(M)).max() < 1e-12      # what makes the test meaningful at this rank and conditioning
    Lbad = L.astype(float)
    Lbad[1, 31, 31] *= 1.0 + 1e-12
    with pytest.raises(AssertionError, match=r"matrix 1, element \(31, 31\) \(8x8 block \(3, 3\)\)"):
        check_L(Lbad, L, M, "perturbed")


def test_rejects_a_transposed_solve():
    M, b = _spd(32, 96, 5)
    L, y, _ = _reference(M, b)
    y_t = backward_ld(L, b)              # L^-T b instead of L^-1 b
    with pytest.raises(AssertionError):
        check_y(y_t.astype(float), y, M, "transposed")


def test_rejects_a_block_left_un_updated():
    M, b = _spd(32, 96, 6, n=1)
    L, _, _ = _reference(M, b)
    check_L(_blocked_cholesky(M[0])[None], L, M, "blocked")
    with pytest.raises(AssertionError, match=r"8x8 block \(3, 2\)"):
        check_L(_blocked_cholesky(M[0], skip=(3, 2, 0))[None], L, M, "block (3, 2) without the update from block column 0")
