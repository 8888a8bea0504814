"""TEST INFRASTRUCTURE ONLY — the unconstrained TVLQR problem as one dense float64 KKT solve.

This is a reference that shares none of the Riccati recursion's assumptions: it writes down the QP
of irs_lqr/tv_lqr.py:69-137 literally and hands its optimality conditions to numpy.linalg.solve.

    minimise   sum_{t<T} (x_t-xd_t)'Q(x_t-xd_t) + 1/2 u_t'R u_t  +  (x_T-xd_T)'Qd(x_T-xd_T)
    over       x_1..x_T, u_0..u_{T-1}          (x_0 fixed)
    s.t.       x_{t+1} = A_t x_t + B_t u_t + c_t

The weights are used exactly as given.  The gradient of (x-d)'W(x-d) is (W + W')(x - d) whatever W
is, so a non-symmetric weight enters through its symmetric part only because calculus says so, not
because this module assumes it.  Sizes: T (2n + m) unknowns; meant for the small and medium problems
of the tests (T (2n + m) up to a few thousand).
"""
import numpy as np


def kkt_system(At, Bt, ct, Q, Qd, R, xd):
    """(KKT matrix, rhs(x0)) of the problem above.  Unknowns: x_1..x_T (T n), u_0..u_{T-1} (T m), then
    the multipliers of the T n dynamics constraints.  rhs accepts x0 [n] or a batch [S, n] and returns
    [D] or [D, S]."""
    At, Bt, ct = (np.asarray(v, dtype=np.float64) for v in (At, Bt, ct))
    Q, Qd, R, xd = (np.asarray(v, dtype=np.float64) for v in (Q, Qd, R, xd))
    T, n, m = At.shape[0], At.shape[1], Bt.shape[2]
    nx, nu = T * n, T * m
    nz = nx + nu
    D = nz + nx
    M = np.zeros((D, D))
    h = np.zeros(nz)
    # objective: Hessian blocks W + W' (W = Q for x_1..x_{T-1}, Qd for x_T, R/2 for every u), gradient
    # offset -(W + W') xd_t.  The x_0 term is a constant.
    for t in range(1, T + 1):
        W = Qd if t == T else Q
        r = (t - 1) * n
        M[r:r + n, r:r + n] = W + W.T
        h[r:r + n] = -(W + W.T).dot(xd[t])
    for t in range(T):
        r = nx + t * m
        M[r:r + m, r:r + m] = 0.5 * (R + R.T)
    # constraints, row block t: x_{t+1} - A_t x_t - B_t u_t = c_t  (x_0 moves to the right-hand side)
    for t in range(T):
        r = nz + t * n
        M[r:r + n, t * n:(t + 1) * n] = np.eye(n)
        if t > 0:
            M[r:r + n, (t - 1) * n:t * n] = -At[t]
        M[r:r + n, nx + t * m:nx + (t + 1) * m] = -Bt[t]
    M[:nz, nz:] = M[nz:, :nz].T

    def rhs(x0):
        x0 = np.asarray(x0, dtype=np.float64)
        batch = x0.ndim == 2
        X0 = x0.T if batch else x0[:, None]
        b = np.zeros((D, X0.shape[1]))
        b[:nz] = -h[:, None]
        b[nz:] = np.tile(ct.reshape(nx, 1), (1, X0.shape[1]))
        b[nz:nz + n] += At[0].dot(X0)
        return b if batch else b[:, 0]

    return M, rhs


def solve(At, Bt, ct, Q, Qd, R, x0, xd):
    """The QP minimiser from x0 [n] -> (x [T+1, n], u [T, m]); x0 [S, n] -> ([S, T+1, n], [S, T, m])."""
    T, n, m = np.shape(At)[0], np.shape(At)[1], np.shape(Bt)[2]
    M, rhs = kkt_system(At, Bt, ct, Q, Qd, R, xd)
    x0 = np.asarray(x0, dtype=np.float64)
    z = np.linalg.solve(M, rhs(x0))
    batch = x0.ndim == 2
    Z = z if batch else z[:, None]
    S = Z.shape[1]
    xs = np.concatenate((x0.reshape(S, 1, n), Z[:T * n].T.reshape(S, T, n)), axis=1)
    us = Z[T * n:T * (n + m)].T.reshape(S, T, m)
    return (xs, us) if batch else (xs[0], us[0])


def gains(At, Bt, ct, Q, Qd, R, xd, t=0):
    """Feedback law of time t, u_t = K_t x_t + k_t, read off the minimiser of the sub-problem that starts at
    t: the minimiser is affine in the start state, so the solves from 0 and from the n unit vectors give
    k_t and the columns of K_t.  -> (K_t [m, n], k_t [m])."""
    n = np.shape(At)[1]
    starts = np.vstack((np.zeros((1, n)), np.eye(n)))
    _, us = solve(At[t:], Bt[t:], ct[t:], Q, Qd, R, starts, xd[t:])
    k = us[0, 0]
    return (us[1:, 0] - k).T, k


def all_gains(At, Bt, ct, Q, Qd, R, xd):
    """K [T, m, n], k [T, m] of every time step (one dense solve per step)."""
    T = np.shape(At)[0]
    out = [gains(At, Bt, ct, Q, Qd, R, xd, t) for t in range(T)]
    return np.stack([o[0] for o in out]), np.stack([o[1] for o in out])


def objective(x, u, xd, Q, Qd, R):
    """The objective above, evaluated literally (terminal weight Qd)."""
    T = u.shape[0]
    e = x - xd[:T + 1]
    c = sum(e[t].dot(Q).dot(e[t]) + 0.5 * u[t].dot(R).dot(u[t]) for t in range(T))
    return c + e[T].dot(Qd).dot(e[T])
