"""CPU pins of the Riccati oracle (oracle/cpu_restatement.py: tvlqr_riccati, solve_tvlqr) on the dense KKT
solve of the literal QP (oracle/dense_lqr.py), for symmetric and for non-symmetric weights.

The cost x'Wx only sees the symmetric part of W, so a non-symmetric Q, Qd or R describes the same
problem as its symmetric part; the recursion must give the minimiser of that problem.  The box oracle
(oracle/box_tvlqr.py) follows the same convention."""
import numpy as np
import pytest

from oracle import box_tvlqr as bq
from oracle import cpu_restatement as cr
from oracle import dense_lqr

DIMS = [(2, 1), (5, 2), (6, 2), (12, 4)]


def rel_err(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


def spd(rng, d, lo=0.5):
    M = rng.standard_normal((d, d))
    return M.dot(M.T) / d + lo * np.eye(d)


def problem(n, m, T, symmetric, seed):
    rng = np.random.default_rng(seed)
    At = np.eye(n) + 0.1 * rng.standard_normal((T, n, n))
    Bt = 0.3 * rng.standard_normal((T, n, m))
    ct = 0.1 * rng.standard_normal((T, n))
    Q, Qd, R = spd(rng, n), 10 * spd(rng, n), spd(rng, m)
    if not symmetric:      # same symmetric parts plus a skew part of comparable size
        Q, Qd, R = (W + (lambda S: S - S.T)(rng.standard_normal(W.shape)) for W in (Q, Qd, R))
    xd = rng.standard_normal((T + 1, n))
    x0 = rng.standard_normal(n)
    return At, Bt, ct, Q, Qd, R, x0, xd


@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("T", [1, 2, 7, 30])
@pytest.mark.parametrize("n,m", DIMS)
def test_riccati_oracle_matches_dense_kkt_solve(n, m, T, symmetric):
    At, Bt, ct, Q, Qd, R, x0, xd = problem(n, m, T, symmetric, seed=100 * n + 10 * m + T)
    xs, us = cr.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd)
    xk, uk = dense_lqr.solve(At, Bt, ct, Q, Qd, R, x0, xd)
    assert rel_err(us, uk) < 1e-10 and rel_err(xs, xk) < 1e-10
    # gains of every step, read off the dense solves of the sub-problems
    K, k = cr.tvlqr_riccati(At, Bt, ct, Q, Qd, R, xd)
    Kk, kk = dense_lqr.all_gains(At, Bt, ct, Q, Qd, R, xd)
    assert rel_err(K, Kk) < 1e-10 and rel_err(k, kk) < 1e-10


@pytest.mark.parametrize("n,m", DIMS)
def test_dense_solve_is_the_minimiser_of_the_literal_objective(n, m):
    """The KKT solution is feasible and no feasible perturbation lowers the objective as written."""
    T = 6
    At, Bt, ct, Q, Qd, R, x0, xd = problem(n, m, T, False, seed=7 * n + m)
    xk, uk = dense_lqr.solve(At, Bt, ct, Q, Qd, R, x0, xd)
    for t in range(T):
        assert np.allclose(xk[t + 1], At[t].dot(xk[t]) + Bt[t].dot(uk[t]) + ct[t], rtol=0, atol=1e-12)
    best = dense_lqr.objective(xk, uk, xd, Q, Qd, R)
    rng = np.random.default_rng(1)
    for _ in range(20):
        u = uk + 1e-3 * rng.standard_normal(uk.shape)
        x = np.zeros_like(xk)
        x[0] = x0
        for t in range(T):
            x[t + 1] = At[t].dot(x[t]) + Bt[t].dot(u[t]) + ct[t]
        assert dense_lqr.objective(x, u, xd, Q, Qd, R) > best


def test_raw_terminal_weight_is_not_the_minimiser():
    """The convention the recursion used before weights were symmetrised (P_T = Qd and the linear terms
    with the raw Q, Qd) gives a different first input than the QP's minimiser: the pins above can tell
    the two apart."""
    n, m, T = 12, 4, 6
    At, Bt, ct, Q, Qd, R, x0, xd = problem(n, m, T, False, seed=3)
    P, p = Qd.copy(), -Qd.dot(xd[T])
    for t in range(T - 1, -1, -1):
        A, B, c = At[t], Bt[t], ct[t]
        w = P.dot(c) + p
        H = 0.5 * R + B.T.dot(P).dot(B)
        H = 0.5 * (H + H.T)
        Kt, kt = -np.linalg.solve(H, B.T.dot(P).dot(A)), -np.linalg.solve(H, B.T.dot(w))
        p = -Q.dot(xd[t]) + A.T.dot(w) + B.T.dot(P).dot(A).T.dot(kt)
        P = Q + A.T.dot(P).dot(A) + B.T.dot(P).dot(A).T.dot(Kt)
        P = 0.5 * (P + P.T)
    u0_raw = Kt.dot(x0) + kt
    _, uk = dense_lqr.solve(At, Bt, ct, Q, Qd, R, x0, xd)
    assert rel_err(u0_raw, uk[0]) > 1e-3


def test_symmetrising_is_a_no_op_for_symmetric_weights():
    """0.5 (W + W') = W exactly for symmetric W, so no stored result of the oracle moves."""
    n, m, T = 6, 2, 9
    At, Bt, ct, Q, Qd, R, x0, xd = problem(n, m, T, True, seed=5)
    Q, Qd, R = (0.5 * (W + W.T) for W in (Q, Qd, R))      # exactly symmetric floats
    K, k = cr.tvlqr_riccati(At, Bt, ct, Q, Qd, R, xd)
    K2, k2, P, H = cr.tvlqr_riccati(At, Bt, ct, Q, Qd, R, xd, return_hessians=True)
    assert np.array_equal(K, K2) and np.array_equal(k, k2) and np.array_equal(P[T], Qd)


def test_box_oracle_uses_the_symmetric_parts():
    """oracle/box_tvlqr.py: augmented gains and the bounded QP of a non-symmetric problem equal those of
    its symmetric part."""
    n, m, T = 5, 2, 8
    At, Bt, ct, Q, Qd, R, x0, xd = problem(n, m, T, False, seed=11)
    Qs, Qds, Rs = (0.5 * (W + W.T) for W in (Q, Qd, R))
    dx, du = bq.penalties(Qs, Rs)
    for a, b in zip(bq.augmented_gains(At, Bt, ct, Q, Qd, R, dx, du), bq.augmented_gains(At, Bt, ct, Qs, Qds, Rs, dx, du)):
        assert np.array_equal(a, b)
    xs, us = dense_lqr.solve(At, Bt, ct, Q, Qd, R, x0, xd)
    lo, hi = np.min(us, axis=0), np.max(us, axis=0)
    ulo, uhi = lo + 0.25 * (hi - lo), hi - 0.25 * (hi - lo)      # active input bounds
    big = 1e6 * np.ones(n)
    x1, u1, _ = bq.admm_box_qp(At, Bt, ct, Q, Qd, R, x0, xd, -big, big, ulo, uhi, dx=dx, du=du)
    x2, u2, _ = bq.admm_box_qp(At, Bt, ct, Qs, Qds, Rs, x0, xd, -big, big, ulo, uhi, dx=dx, du=du)
    assert np.array_equal(u1, u2) and np.array_equal(x1, x2)
    xr, ur, res = bq.dense_qp_reference(At, Bt, ct, Q, Qd, R, x0, xd, -big, big, ulo, uhi)
    assert res.success
    np.testing.assert_allclose(u1, ur, rtol=0, atol=2e-5)
