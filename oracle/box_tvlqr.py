"""TEST INFRASTRUCTURE ONLY — float64 numpy restatement of the box-constrained TVLQR.

The reference solves, at every timestep t0 of IrsLqr.local_descent (irs_lqr/irs_lqr.py:169-184), the
QP of irs_lqr/tv_lqr.py:69-137 over the remaining horizon with absolute box bounds on states and
inputs (:113-118, :132-134) through Drake + OSQP (an ADMM solver; version unpinned, not installable
here) and applies the first input to the true dynamics.  PARITY UNPINNED against the reference's
numbers: there is no stored result that isolates a bounded solve, and OSQP stops at 1e-3.  What is
pinned instead: the QP itself.  `admm_box_qp` below solves exactly that QP (unique minimiser: the
cost is strictly convex in u and the constraints are convex) by ADMM on the box split, with the
equality-constrained step done by the affine Riccati recursion; tests check its output against an
independent dense QP solve (scipy) and the CUDA kernel against it.

Split:  minimise f(y) + g(z) s.t. y = z,  y = (x_1..x_H, u_0..u_{H-1}),
        f = QP cost + indicator(dynamics from the fixed x_0),  g = indicator(box).
Penalty D = diag(dx) on states, diag(du) on inputs; scaled dual w; over-relaxation alpha.
"""
import numpy as np

DEFAULT_RHO0 = 1.0
DEFAULT_ALPHA = 1.6
DEFAULT_EPS = 1e-10
DEFAULT_MAX_ITER = 100000


def _sym(W):
    """The symmetric part of a weight: x'Wx sees nothing else (for symmetric W exactly W)."""
    W = np.asarray(W, dtype=np.float64)
    return 0.5 * (W + W.T)


def penalties(Q, R, rho0=DEFAULT_RHO0):
    """Per-coordinate ADMM penalties: rho0 times the cost curvature of the coordinate, floored at
    the mean curvature (coordinates with zero weight still get a usable penalty)."""
    qd, rd = np.diag(Q).copy(), 0.5 * np.diag(R)
    dx = rho0 * np.maximum(qd, qd.mean())
    du = rho0 * np.maximum(rd, rd.mean())
    return dx, du


def augmented_gains(At, Bt, ct, Q, Qd, R, dx, du):
    """Matrix part of the Riccati recursion for the augmented cost (independent of z, w and of the
    start time): K_t, Hinv_t, P_t (t = 0..T)."""
    T, n, m = At.shape[0], Q.shape[0], R.shape[0]
    Q, Qd, R = _sym(Q), _sym(Qd), _sym(R)
    Qe, Qde, Re = Q + 0.5 * np.diag(dx), Qd + 0.5 * np.diag(dx), 0.5 * R + 0.5 * np.diag(du)
    K = np.zeros((T, m, n))
    Hinv = np.zeros((T, m, m))
    P = np.zeros((T + 1, n, n))
    P[T] = Qde
    for t in range(T - 1, -1, -1):
        A, B = At[t], Bt[t]
        PA, PB = P[t + 1].dot(A), P[t + 1].dot(B)
        H = Re + B.T.dot(PB)
        H = 0.5 * (H + H.T)
        Hinv[t] = np.linalg.inv(H)
        G = B.T.dot(PA)
        K[t] = -Hinv[t].dot(G)
        Pn = Qe + A.T.dot(PA) + G.T.dot(K[t])
        P[t] = 0.5 * (Pn + Pn.T)
    return K, Hinv, P


def admm_box_qp(At, Bt, ct, Q, Qd, R, x0, xd, xlo, xhi, ulo, uhi, gains=None, dx=None, du=None,
                z=None, w=None, t0=0, alpha=DEFAULT_ALPHA, eps=DEFAULT_EPS, max_iter=DEFAULT_MAX_ITER):
    """QP over the horizon t0..T from the fixed state x0 = x_{t0}.  Arrays are indexed by ABSOLUTE
    time (zx[t], wx[t] for t0 < t <= T; zu[t], wu[t] for t0 <= t < T) so that consecutive MPC solves
    warm-start each other.  Returns (x[T+1,n], u[T,m], iterations); entries before t0 are untouched
    zeros.  Bounds are per coordinate (constant in time), as IrsLqr passes them (irs_lqr.py:160-167);
    the bound on the fixed x_{t0} is not part of the problem."""
    T, n, m = At.shape[0], Q.shape[0], R.shape[0]
    Q, Qd = _sym(Q), _sym(Qd)
    if dx is None:
        dx, du = penalties(Q, R)
    if gains is None:
        gains = augmented_gains(At, Bt, ct, Q, Qd, R, dx, du)
    K, Hinv, P = gains
    if z is None:
        z = (np.zeros((T + 1, n)), np.zeros((T, m)))
        w = (np.zeros((T + 1, n)), np.zeros((T, m)))
        cold = True
    else:
        cold = False
    zx, zu = z
    wx, wu = w
    x = np.zeros((T + 1, n))
    u = np.zeros((T, m))
    kk = np.zeros((T, m))
    p = np.zeros((T + 1, n))
    x[t0] = x0
    Pc = np.einsum("tij,tj->ti", P[1:], ct)          # P_{t+1} c_t
    if cold:
        # start from the projection of the unconstrained-looking iterate: z = clip(0-penalty solve)
        zx[:] = np.clip(xd[:T + 1], xlo, xhi)
        zu[:] = np.clip(0.0, ulo, uhi)
    for it in range(1, max_iter + 1):
        # backward vectors
        p[T] = -(Qd.dot(xd[T]) + 0.5 * dx * (zx[T] - wx[T]))
        for t in range(T - 1, t0 - 1, -1):
            ww = Pc[t] + p[t + 1]
            ru = 0.5 * du * (zu[t] - wu[t])
            g = Bt[t].T.dot(ww) - ru
            kk[t] = -Hinv[t].dot(g)
            if t > t0:
                qx = Q.dot(xd[t]) + 0.5 * dx * (zx[t] - wx[t])
                p[t] = -qx + At[t].T.dot(ww) + K[t].T.dot(g)
        # forward
        for t in range(t0, T):
            u[t] = K[t].dot(x[t]) + kk[t]
            x[t + 1] = At[t].dot(x[t]) + Bt[t].dot(u[t]) + ct[t]
        # relaxed projection + dual
        xh = alpha * x[t0 + 1:] + (1.0 - alpha) * zx[t0 + 1:]
        uh = alpha * u[t0:] + (1.0 - alpha) * zu[t0:]
        # boxes: [n] / [m] constant over the horizon, or one row per timestep ([T+1, n] / [T, m])
        zx_new = np.clip(xh + wx[t0 + 1:], xlo[t0 + 1:] if np.ndim(xlo) == 2 else xlo,
                         xhi[t0 + 1:] if np.ndim(xhi) == 2 else xhi)
        zu_new = np.clip(uh + wu[t0:], ulo[t0:] if np.ndim(ulo) == 2 else ulo, uhi[t0:] if np.ndim(uhi) == 2 else uhi)
        wx[t0 + 1:] += xh - zx_new
        wu[t0:] += uh - zu_new
        r_prim = max(np.max(np.abs(x[t0 + 1:] - zx_new)), np.max(np.abs(u[t0:] - zu_new)))
        # residuals in the units of z (tvlqr_box.cuh): the test is invariant under a scaling of the weights
        r_dual = max(np.max(np.abs(zx_new - zx[t0 + 1:])), np.max(np.abs(zu_new - zu[t0:])))
        scale = max(1.0, np.max(np.abs(zx_new)), np.max(np.abs(zu_new)))
        zx[t0 + 1:] = zx_new
        zu[t0:] = zu_new
        if r_prim <= eps * scale and r_dual <= eps * scale:
            return x, u, it
    raise ValueError("TV_LQR failed. Optimization problem is not solved.")


def mpc_box_descent(system, At, Bt, ct, Q, Qd, R, x0, xd, xlo, xhi, ulo, uhi, rho0=DEFAULT_RHO0,
                    alpha=DEFAULT_ALPHA, eps=DEFAULT_EPS, max_iter=DEFAULT_MAX_ITER, gains0=None, tol=1e-9):
    """IrsLqr.local_descent's loop (irs_lqr.py:169-184) with the bounded QP: at every t0 solve over
    the remaining horizon from the ACTUAL state, apply the first input (the feasible split variable
    z_u) to the true dynamics.  gains0 = (K0, k0), the unconstrained Riccati gains: a start time whose
    unconstrained plan stays inside the box has inactive bounds, its QP minimiser is K0 x + k0 and the
    ADMM is skipped (exactly what a QP solver returns there).  Returns (x_trj, u_trj, total ADMM
    iterations)."""
    T, n, m = At.shape[0], Q.shape[0], R.shape[0]
    dx, du = penalties(Q, R, rho0)
    gains = augmented_gains(At, Bt, ct, Q, Qd, R, dx, du)
    z = (np.zeros((T + 1, n)), np.zeros((T, m)))
    w = (np.zeros((T + 1, n)), np.zeros((T, m)))
    z[0][:] = np.clip(xd[:T + 1], xlo, xhi)
    z[1][:] = np.clip(0.0, ulo, uhi)
    x_trj = np.zeros((T + 1, n))
    u_trj = np.zeros((T, m))
    x_trj[0] = x0
    total = 0
    for t0 in range(T):
        if gains0 is not None:
            K0, k0 = gains0
            xs, ok, u_first = x_trj[t0], True, None
            for t in range(t0, T):
                us = K0[t].dot(xs) + k0[t]
                if u_first is None:
                    u_first = us
                xs = At[t].dot(xs) + Bt[t].dot(us) + ct[t]
                if np.any(us < ulo - tol) or np.any(us > uhi + tol) or np.any(xs < xlo - tol) or np.any(xs > xhi + tol):
                    ok = False
                    break
            if ok:
                u_trj[t0] = u_first
                x_trj[t0 + 1] = system.dynamics(x_trj[t0], u_trj[t0])
                continue
        _, _, it = admm_box_qp(At, Bt, ct, Q, Qd, R, x_trj[t0], xd, xlo, xhi, ulo, uhi, gains, dx, du, z, w,
                               t0=t0, alpha=alpha, eps=eps, max_iter=max_iter)
        total += it
        u_trj[t0] = z[1][t0]
        x_trj[t0 + 1] = system.dynamics(x_trj[t0], u_trj[t0])
    return x_trj, u_trj, total


def dense_qp_reference(At, Bt, ct, Q, Qd, R, x0, xd, xlo, xhi, ulo, uhi):
    """Independent check of admm_box_qp on SMALL horizons: condense the states out
    (x = Sx x0 + Su u + s0) and solve the inequality-constrained QP in u with scipy (SLSQP)."""
    from scipy.optimize import minimize
    T, n, m = At.shape[0], Q.shape[0], R.shape[0]
    Q, Qd, R = _sym(Q), _sym(Qd), _sym(R)      # the gradient below assumes symmetric weights
    Su = np.zeros(((T + 1) * n, T * m))
    s0 = np.zeros((T + 1) * n)
    s0[:n] = x0
    for t in range(T):
        r0, r1 = t * n, (t + 1) * n
        s0[r1:r1 + n] = At[t].dot(s0[r0:r1]) + ct[t]
        Su[r1:r1 + n] = At[t].dot(Su[r0:r1])
        Su[r1:r1 + n, t * m:(t + 1) * m] += Bt[t]
    Qbig = np.zeros(((T + 1) * n, (T + 1) * n))
    for t in range(T):
        Qbig[t * n:(t + 1) * n, t * n:(t + 1) * n] = Q
    Qbig[T * n:, T * n:] = Qd
    Rbig = np.kron(np.eye(T), 0.5 * R)
    xdv = xd[:T + 1].reshape(-1)

    def cost(uv):
        e = s0 + Su.dot(uv) - xdv
        return e.dot(Qbig).dot(e) + uv.dot(Rbig).dot(uv)

    def grad(uv):
        e = s0 + Su.dot(uv) - xdv
        return 2.0 * Su.T.dot(Qbig.dot(e)) + 2.0 * Rbig.dot(uv)

    # boxes: [n] / [m] constant over the horizon, or one row per timestep ([T+1, n] / [T, m])
    lo = np.asarray(xlo)[1:T + 1].reshape(-1) if np.ndim(xlo) == 2 else np.tile(xlo, T)
    hi = np.asarray(xhi)[1:T + 1].reshape(-1) if np.ndim(xhi) == 2 else np.tile(xhi, T)
    cons = [{"type": "ineq", "fun": lambda uv: (s0 + Su.dot(uv))[n:] - lo, "jac": lambda uv: Su[n:]},
            {"type": "ineq", "fun": lambda uv: hi - (s0 + Su.dot(uv))[n:], "jac": lambda uv: -Su[n:]}]
    bounds = list(zip(np.asarray(ulo)[:T].reshape(-1) if np.ndim(ulo) == 2 else np.tile(ulo, T),
                      np.asarray(uhi)[:T].reshape(-1) if np.ndim(uhi) == 2 else np.tile(uhi, T)))
    res = minimize(cost, np.zeros(T * m), jac=grad, bounds=bounds, constraints=cons, method="SLSQP",
                   options={"maxiter": 500, "ftol": 1e-14})
    uv = res.x
    return (s0 + Su.dot(uv)).reshape(T + 1, n), uv.reshape(T, m), res
