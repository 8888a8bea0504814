"""TEST INFRASTRUCTURE ONLY — float64 numpy restatement of the iRS-MPC hot path.

This module is the *checker* for the CUDA path.  Only `tests/`, `__graft_entry__.smoke()` and the
`cpu_baseline` / `--impl reference` legs of `bench.py` may import it; the product package
`irs_mpc_b200` never does (it fails loudly when the CUDA library is missing instead).

Every function cites the reference lines (relative to /root/reference) it restates.  Pinning
status (see tests/test_oracle_golden.py and tests/golden/):

* dynamics / dynamics_batch / projection / rollout / evaluate_cost / zero-order get_TV_matrices:
  pinned against outputs of the reference's own code (run under oracle/ref_import.py, vectors
  committed under tests/golden/ by oracle/make_golden.py).
* jacobian_xu (pydrake.symbolic / forwarddiff in the reference — cannot run here): analytic
  forms, pinned indirectly through the stored exact-variant cost curves
  examples/pendulum/analysis/pendulum_exact.csv and examples/quadrotor/analysis/quadrotor_exact.csv
  and cross-checked against complex-step differentiation of the pinned dynamics.
* solve_tvlqr (pydrake MathematicalProgram + OSQP, version unpinned, not installed): restated as
  the equivalent affine Riccati recursion (valid while the box bounds are inactive), pinned on the
  same two CSVs.  Bicycle (active steer bound) is *parity unpinned* beyond entry 0.
"""
import time

import numpy as np


# ----------------------------------------------------------------------------------------------
# Dynamical systems (float64).  All take/return numpy arrays; *_batch are vectorised over rows.
# ----------------------------------------------------------------------------------------------
class PendulumOracle:
    """examples/pendulum/pendulum_dynamics.py:8-127 (n=2, m=1, semi-implicit Euler)."""

    dim_x, dim_u = 2, 1

    def __init__(self, h):
        self.h = h

    def dynamics_batch(self, x, u):
        # pendulum_dynamics.py:62-81
        x = np.asarray(x)
        u = np.asarray(u)
        v_next = x[:, 1] + self.h * (u[:, 0] - np.sin(x[:, 0]))
        th_next = x[:, 0] + self.h * v_next
        return np.stack((th_next, v_next), axis=1)

    def dynamics(self, x, u):
        # pendulum_dynamics.py:46-60
        return self.dynamics_batch(np.asarray(x)[None], np.asarray(u)[None])[0]

    def jacobian_xu_batch(self, x, u):
        # pendulum_dynamics.py:110-127 (symbolic Jacobian of :28-43, evaluated per sample)
        x = np.asarray(x)
        h = self.h
        c = np.cos(x[:, 0])
        J = np.zeros((x.shape[0], 2, 3))
        J[:, 0, 0] = 1.0 - h * h * c
        J[:, 0, 1] = h
        J[:, 0, 2] = h * h
        J[:, 1, 0] = -h * c
        J[:, 1, 1] = 1.0
        J[:, 1, 2] = h
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None], np.asarray(u)[None])[0]


class BicycleOracle:
    """examples/bicycle/bicycle_dynamics.py:8-132 (n=5, m=2, explicit Euler)."""

    dim_x, dim_u = 5, 2

    def __init__(self, h):
        self.h = h

    def dynamics_batch(self, x, u):
        # bicycle_dynamics.py:66-86
        x = np.asarray(x)
        u = np.asarray(u)
        th, v, de = x[:, 2], x[:, 3], x[:, 4]
        rate = np.stack((v * np.cos(th), v * np.sin(th), v * np.tan(de), u[:, 0], u[:, 1]), axis=1)
        return x + self.h * rate

    def dynamics(self, x, u):
        # bicycle_dynamics.py:47-64
        return self.dynamics_batch(np.asarray(x)[None], np.asarray(u)[None])[0]

    def jacobian_xu_batch(self, x, u):
        # bicycle_dynamics.py:115-132 (symbolic Jacobian of :26-44)
        x = np.asarray(x)
        h = self.h
        th, v, de = x[:, 2], x[:, 3], x[:, 4]
        J = np.zeros((x.shape[0], 5, 7))
        J[:, np.arange(5), np.arange(5)] = 1.0
        J[:, 0, 2] = -h * v * np.sin(th)
        J[:, 0, 3] = h * np.cos(th)
        J[:, 1, 2] = h * v * np.cos(th)
        J[:, 1, 3] = h * np.sin(th)
        J[:, 2, 3] = h * np.tan(de)
        J[:, 2, 4] = h * v / np.cos(de) ** 2
        J[:, 3, 5] = h
        J[:, 4, 6] = h
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None], np.asarray(u)[None])[0]


class QuadrotorOracle:
    """examples/quadrotor/quadrotor_dynamics.py:15-231 (n=12, m=4, rpy Euler angles, explicit Euler).

    x = [xyz, rpy, xyz_dot, rpy_dot]; constants from :26-38.
    """

    dim_x, dim_u = 12, 4

    def __init__(self, h):
        self.h = h
        self.m = 0.775
        self.L = 0.15
        self.g = 9.81
        self.Idiag = np.array([0.0015, 0.0025, 0.0035])
        self.kF = 1.0
        self.kM = 0.0245

    def _xdot(self, x, u):
        """Vectorised restatement of quadrotor_dynamics.py:40-77 with helpers :150-231 inlined.

        Works for float64 and complex128 (the latter is used for complex-step Jacobians).
        """
        uF = self.kF * u
        uM = self.kM * u
        Fz = uF[:, 0] + uF[:, 1] + uF[:, 2] + uF[:, 3]                       # :44
        M0 = self.L * (-uF[:, 0] - uF[:, 1] + uF[:, 2] + uF[:, 3])           # :45
        M1 = self.L * (-uF[:, 0] - uF[:, 3] + uF[:, 1] + uF[:, 2])           # :46
        M2 = -uM[:, 0] + uM[:, 1] - uM[:, 2] + uM[:, 3]                      # :47
        ro, pi_, ya = x[:, 3], x[:, 4], x[:, 5]
        rd = x[:, 9:12]
        sr, cr = np.sin(ro), np.cos(ro)
        sp, cp = np.sin(pi_), np.cos(pi_)
        sy, cy = np.sin(ya), np.cos(ya)
        # Third column of R_WB = Rz(yaw) Ry(pitch) Rx(roll) (:150-189); F has only a z component.
        r13 = cy * sp * cr + sy * sr
        r23 = sy * sp * cr - cy * sr
        r33 = cp * cr
        inv_m = 1.0 / self.m
        acc = np.stack((inv_m * (r13 * Fz), inv_m * (r23 * Fz),
                        inv_m * (r33 * Fz - self.m * self.g)), axis=1)      # :54
        # pqr = PhiInv(rpy) rpy_d (:57-58, :191-202)
        p = rd[:, 0] - sp * rd[:, 2]
        q = cr * rd[:, 1] + sr * cp * rd[:, 2]
        r = -sr * rd[:, 1] + cr * cp * rd[:, 2]
        I0, I1, I2 = self.Idiag
        # pqr_d = I^-1 (M - pqr x (I pqr)) (:59)
        pd = (M0 - (q * (I2 * r) - r * (I1 * q))) / I0
        qd = (M1 - (r * (I0 * p) - p * (I2 * r))) / I1
        rdd = (M2 - (p * (I1 * q) - q * (I0 * p))) / I2
        # Phi (:204-215) and its time derivative PhiD . rpy_d (:218-231)
        tp = sp / cp
        cp2 = cp * cp
        d_roll, d_pitch = rd[:, 0], rd[:, 1]
        Phi01, Phi02 = sr * tp, cr * tp
        Phi21, Phi22 = sr / cp, cr / cp
        dPhi01 = cr * tp * d_roll + sr / cp2 * d_pitch
        dPhi02 = -sr * tp * d_roll + cr / cp2 * d_pitch
        dPhi11 = -sr * d_roll
        dPhi12 = -cr * d_roll
        dPhi21 = cr / cp * d_roll + sr * sp / cp2 * d_pitch
        dPhi22 = -sr / cp * d_roll + cr * sp / cp2 * d_pitch
        # rpy_dd = Phi pqr_d + (PhiD . rpy_d) pqr (:68)
        a0 = pd + Phi01 * qd + Phi02 * rdd + dPhi01 * q + dPhi02 * r
        a1 = cr * qd - sr * rdd + dPhi11 * q + dPhi12 * r
        a2 = Phi21 * qd + Phi22 * rdd + dPhi21 * q + dPhi22 * r
        ang = np.stack((a0, a1, a2), axis=1)
        return np.concatenate((x[:, 6:12], acc, ang), axis=1)              # :70-72

    def dynamics_batch(self, x, u):
        # quadrotor_dynamics.py:79-91 (a Python loop over :40-77 in the reference)
        x = np.asarray(x)
        u = np.asarray(u)
        return x + self.h * self._xdot(x, u)

    def dynamics(self, x, u):
        return self.dynamics_batch(np.asarray(x)[None], np.asarray(u)[None])[0]

    def jacobian_xu_batch(self, x, u):
        """quadrotor_dynamics.py:132-148 uses pydrake.forwarddiff (exact AD).  Restated with
        complex-step differentiation (exact to round-off for analytic functions)."""
        x = np.asarray(x, dtype=np.float64)
        u = np.asarray(u, dtype=np.float64)
        B = x.shape[0]
        eps = 1e-30
        J = np.zeros((B, 12, 16))
        for k in range(16):
            xc = x.astype(np.complex128)
            uc = u.astype(np.complex128)
            if k < 12:
                xc[:, k] += 1j * eps
            else:
                uc[:, k - 12] += 1j * eps
            J[:, :, k] = np.imag(xc + self.h * self._xdot(xc, uc)) / eps
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None], np.asarray(u)[None])[0]


class ThreeCartOracle:
    """examples/three_cart/three_cart_dynamics.py:8-264 (n=6, m=2, inelastic 1-D contact).

    NOTE the reference's `dynamics` (:22-107) and `dynamics_batch` (:109-194) DISAGREE in the
    pair-collision cases: the scalar version pushes each cart out by half the penetration depth
    (:68-69, :84-85), the batch version by the full depth (:175-176, :187-188).  Both are restated
    faithfully; the zero-order fit mixes them (irs_lqr_zero_order.py:51-52).
    """

    dim_x, dim_u = 6, 2

    def __init__(self, dt):
        self.h = dt
        self.d = 0.2

    def _free_step(self, x, u):
        # :33-41 / :130-141
        h = self.h
        v1 = x[:, 3] + h * u[:, 0]
        v2 = x[:, 4].copy()
        v3 = x[:, 5] + h * u[:, 1]
        q1 = x[:, 0] + h * v1
        q2 = x[:, 1] + h * v2
        q3 = x[:, 2] + h * v3
        return np.stack((q1, q2, q3, v1, v2, v3), axis=1)

    def _resolve(self, s, pair_factor, fix_velocity):
        """Contact resolution shared by dynamics / dynamics_batch / projection.

        pair_factor: 0.5 (scalar dynamics :68-69,:84-85 and projection :241-242,:258-259) or
        1.0 (dynamics_batch :175-176,:187-188)."""
        d = self.d
        g12 = s[:, 1] - s[:, 0] < d
        g23 = s[:, 2] - s[:, 1] < d
        both = g12 & g23
        only12 = g12 & ~g23
        only23 = ~g12 & g23
        out = s.copy()
        # all three (:49-63 / :159-169 / :222-228): positions -> mean +- d, velocities -> mean
        mid = np.mean(s[both][:, 0:3], axis=1)
        out[both, 1] = mid
        out[both, 0] = mid - d
        out[both, 2] = mid + d
        if fix_velocity:
            vavg = np.mean(s[both][:, 3:6], axis=1)
            out[both, 3] = vavg
            out[both, 4] = vavg
            out[both, 5] = vavg
        # carts 1,2 (:65-78 / :171-181 / :237-244)
        depth = d - (s[only12, 1] - s[only12, 0])
        out[only12, 1] = s[only12, 1] + pair_factor * depth
        out[only12, 0] = s[only12, 0] - pair_factor * depth
        if fix_velocity:
            vavg = np.mean(s[only12][:, 3:5], axis=1)
            out[only12, 3] = vavg
            out[only12, 4] = vavg
        # carts 2,3 (:80-94 / :183-192 / :254-261)
        depth = d - (s[only23, 2] - s[only23, 1])
        out[only23, 2] = s[only23, 2] + pair_factor * depth
        out[only23, 1] = s[only23, 1] - pair_factor * depth
        if fix_velocity:
            vavg = np.mean(s[only23][:, 4:6], axis=1)
            out[only23, 4] = vavg
            out[only23, 5] = vavg
        return out

    def dynamics_batch(self, x, u):
        # :109-194 (full-depth push-out in pair cases)
        s = self._free_step(np.asarray(x, dtype=np.float64), np.asarray(u, dtype=np.float64))
        return self._resolve(s, 1.0, True)

    def dynamics_scalar_batch(self, x, u):
        """Row-wise application of the *scalar* `dynamics` (:22-107): half-depth push-out.

        np.mean over three numbers in :159-166 vs (1./3.)*(a+b+c) in :52/:60 differ by <=1ulp;
        the scalar form is restated literally here."""
        s = self._free_step(np.asarray(x, dtype=np.float64), np.asarray(u, dtype=np.float64))
        d = self.d
        g12 = s[:, 1] - s[:, 0] < d
        g23 = s[:, 2] - s[:, 1] < d
        both = g12 & g23
        only12 = g12 & ~g23
        only23 = ~g12 & g23
        out = s.copy()
        mid = (1. / 3.) * (s[both, 0] + s[both, 1] + s[both, 2])
        out[both, 1] = mid
        out[both, 0] = mid - d
        out[both, 2] = mid + d
        vavg = (1. / 3.) * (s[both, 3] + s[both, 4] + s[both, 5])
        out[both, 3] = vavg
        out[both, 4] = vavg
        out[both, 5] = vavg
        depth = d - (s[only12, 1] - s[only12, 0])
        out[only12, 1] = s[only12, 1] + 0.5 * depth
        out[only12, 0] = s[only12, 0] - 0.5 * depth
        vavg = 0.5 * (s[only12, 3] + s[only12, 4])
        out[only12, 3] = vavg
        out[only12, 4] = vavg
        depth = d - (s[only23, 2] - s[only23, 1])
        out[only23, 2] = s[only23, 2] + 0.5 * depth
        out[only23, 1] = s[only23, 1] - 0.5 * depth
        vavg = 0.5 * (s[only23, 4] + s[only23, 5])
        out[only23, 4] = vavg
        out[only23, 5] = vavg
        return out

    def dynamics(self, x, u):
        return self.dynamics_scalar_batch(np.asarray(x)[None], np.asarray(u)[None])[0]

    def contact_case(self, x, u):
        """Integer case id per row (0 none, 1 all three, 2 carts 1-2, 3 carts 2-3) — the
        sample bookkeeping that must match bit-for-bit (:146-157)."""
        s = self._free_step(np.asarray(x, dtype=np.float64), np.asarray(u, dtype=np.float64))
        g12 = s[:, 1] - s[:, 0] < self.d
        g23 = s[:, 2] - s[:, 1] < self.d
        return (np.where(g12 & g23, 1, 0) + np.where(g12 & ~g23, 2, 0)
                + np.where(~g12 & g23, 3, 0)).astype(np.int32)

    def projection(self, x, dx, u, du):
        """:196-264 — returns ABSOLUTE points (x+dx projected, u+du).  The reference evaluates the
        three masks sequentially on the partially projected array (:216,:232,:249); after the
        all-three case the gaps are exactly d up to one rounding, so re-evaluating can move a
        sample by at most ~1e-16.  Restated sequentially to match."""
        xp = np.asarray(x, dtype=np.float64) + np.asarray(dx, dtype=np.float64)
        up = np.asarray(u, dtype=np.float64) + np.asarray(du, dtype=np.float64)
        d = self.d
        m = (xp[:, 1] - xp[:, 0] < d) & (xp[:, 2] - xp[:, 1] < d)
        mid = np.mean(xp[m][:, 0:3], axis=1)
        xp[m, 1] = mid
        xp[m, 0] = mid - d
        xp[m, 2] = mid + d
        m = (xp[:, 1] - xp[:, 0] < d) & (xp[:, 2] - xp[:, 1] >= d)
        depth = d - (xp[m, 1] - xp[m, 0])
        xp[m, 1] += 0.5 * depth
        xp[m, 0] -= 0.5 * depth
        m = (xp[:, 1] - xp[:, 0] >= d) & (xp[:, 2] - xp[:, 1] < d)
        depth = d - (xp[m, 2] - xp[m, 1])
        xp[m, 2] += 0.5 * depth
        xp[m, 1] -= 0.5 * depth
        return xp, up


SYSTEMS = {
    "pendulum": PendulumOracle,
    "bicycle": BicycleOracle,
    "quadrotor": QuadrotorOracle,
    "three_cart": ThreeCartOracle,
}


# ----------------------------------------------------------------------------------------------
# Solver pieces
# ----------------------------------------------------------------------------------------------
def rollout(system, x0, u_trj):
    """irs_lqr/irs_lqr.py:105-119 — open-loop rollout with the scalar `dynamics`."""
    T = u_trj.shape[0]
    x_trj = np.zeros((T + 1, system.dim_x))
    x_trj[0] = x0
    for t in range(T):
        x_trj[t + 1] = system.dynamics(x_trj[t], u_trj[t])
    return x_trj


def evaluate_cost(x_trj, u_trj, xd_trj, Q, R):
    """irs_lqr/irs_lqr.py:121-137 — NOTE the terminal term uses Q, not Qd (:135-136)."""
    T = u_trj.shape[0]
    e = x_trj[:T] - xd_trj[:T]
    cost = 0.0
    for t in range(T):
        cost += e[t].dot(Q).dot(e[t])
        cost += u_trj[t].dot(R).dot(u_trj[t])
    eT = x_trj[T] - xd_trj[T]
    cost += eT.dot(Q).dot(eT)
    return cost


def affine_offset(system, A, B, xbar, ubar):
    """c_t = f(xbar,ubar) - A xbar - B ubar with the *scalar* nominal dynamics
    (irs_lqr_zero_order.py:61-62, irs_lqr_first_order.py:52-53, irs_lqr_exact.py:29-30)."""
    return system.dynamics(xbar, ubar) - A.dot(xbar) - B.dot(ubar)


def least_squares_AB(dxdu, deltaf, dim_x):
    """irs_lqr_zero_order.py:27-36 — lstsq without intercept column, default rcond."""
    AB = np.linalg.lstsq(dxdu, deltaf, rcond=None)[0].T
    return AB[:, :dim_x], AB[:, dim_x:]


def zero_order_tv_matrices(system, x_trj, u_trj, deltas):
    """irs_lqr_zero_order.py:38-63 with the sampled deltas supplied explicitly.

    deltas: array [T, N, n+m] holding what `sampling(xbar, ubar, iter)` returned for step t
    (dx in the first n columns, du in the last m)."""
    T = u_trj.shape[0]
    n, m = system.dim_x, system.dim_u
    At = np.zeros((T, n, n))
    Bt = np.zeros((T, n, m))
    ct = np.zeros((T, n))
    for t in range(T):
        dx = deltas[t][:, :n]
        du = deltas[t][:, n:]
        fdt = system.dynamics_batch(x_trj[t] + dx, u_trj[t] + du)    # :51 (batch variant)
        ft = system.dynamics(x_trj[t], u_trj[t])                     # :52 (scalar variant)
        At[t], Bt[t] = least_squares_AB(np.hstack((dx, du)), fdt - ft, n)
        ct[t] = affine_offset(system, At[t], Bt[t], x_trj[t], u_trj[t])
    return At, Bt, ct


def first_order_tv_matrices(system, x_trj, u_trj, deltas):
    """irs_lqr_first_order.py:28-54 — mean over samples of the Jacobian at the perturbed points."""
    T = u_trj.shape[0]
    n, m = system.dim_x, system.dim_u
    At = np.zeros((T, n, n))
    Bt = np.zeros((T, n, m))
    ct = np.zeros((T, n))
    for t in range(T):
        dx = deltas[t][:, :n]
        du = deltas[t][:, n:]
        J = np.mean(system.jacobian_xu_batch(x_trj[t] + dx, u_trj[t] + du), axis=0)   # :46-48
        At[t], Bt[t] = J[:, :n], J[:, n:]
        ct[t] = affine_offset(system, At[t], Bt[t], x_trj[t], u_trj[t])
    return At, Bt, ct


def exact_tv_matrices(system, x_trj, u_trj):
    """irs_lqr_exact.py:15-31 — Jacobian at the nominal point."""
    T = u_trj.shape[0]
    n, m = system.dim_x, system.dim_u
    At = np.zeros((T, n, n))
    Bt = np.zeros((T, n, m))
    ct = np.zeros((T, n))
    for t in range(T):
        J = system.jacobian_xu(x_trj[t], u_trj[t])
        At[t], Bt[t] = J[:, :n], J[:, n:]
        ct[t] = affine_offset(system, At[t], Bt[t], x_trj[t], u_trj[t])
    return At, Bt, ct


def tvlqr_riccati(At, Bt, ct, Q, Qd, R, xd_trj, return_hessians=False):
    """Backward pass equivalent to the QP of irs_lqr/tv_lqr.py:69-137 when no bound is active.

    Cost restated from the QP: sum_{s<T} (x_s-xd_s)'Q(x_s-xd_s) + (1/2) u_s'R u_s  (:110, :127;
    Drake's AddQuadraticCost(Q,b,x) is 0.5 x'Qx + b'x) + (x_T-xd_T)'Qd(x_T-xd_T) (:130), subject to
    x_{s+1} = A_s x_s + B_s u_s + c_s (:92-95).  Value function V_s(x) = x'P_s x + 2 p_s'x + const.
    The cost only sees the symmetric parts of Q, Qd and R, so the recursion runs on those (for symmetric
    weights 0.5 (W + W') = W exactly).
    Returns feedback gains K[T,m,n], k[T,m] with u_s = K_s x_s + k_s; with return_hessians also the
    value-function Hessians P[T+1,n,n] and the step Hessians H[T,m,m] = R/2 + B'P_{s+1}B.
    """
    T = At.shape[0]
    n = Q.shape[0]
    m = R.shape[0]
    Q, Qd, R = 0.5 * (Q + Q.T), 0.5 * (Qd + Qd.T), 0.5 * (R + R.T)
    Rh = 0.5 * R
    K = np.zeros((T, m, n))
    k = np.zeros((T, m))
    Ps = np.zeros((T + 1, n, n))
    Hs = np.zeros((T, m, m))
    P = Qd.copy()
    p = -Qd.dot(xd_trj[T])
    Ps[T] = P
    for t in range(T - 1, -1, -1):
        A, B, c = At[t], Bt[t], ct[t]
        PA = P.dot(A)
        PB = P.dot(B)
        w = P.dot(c) + p
        H = Rh + B.T.dot(PB)
        G = B.T.dot(PA)
        g = B.T.dot(w)
        Hs[t] = H
        L = np.linalg.cholesky(H)          # raises LinAlgError if H is not SPD
        Kt = -np.linalg.solve(L.T, np.linalg.solve(L, G))
        kt = -np.linalg.solve(L.T, np.linalg.solve(L, g))
        K[t], k[t] = Kt, kt
        p = -Q.dot(xd_trj[t]) + A.T.dot(w) + G.T.dot(kt)
        P = Q + A.T.dot(PA) + G.T.dot(Kt)
        P = 0.5 * (P + P.T)
        Ps[t] = P
    if return_hessians:
        return K, k, Ps, Hs
    return K, k


def solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, x_trj_d, solver=None, indices_u_into_x=None,
                x_bound_abs=None, u_bound_abs=None, x_bound_rel=None, u_bound_rel=None,
                xinit=None, uinit=None, bound_tol=1e-9):
    """irs_lqr/tv_lqr.py:30-145 restated for the in-scope argument set (indices_u_into_x None,
    relative bounds None).  Returns the QP minimiser (x*[T+1,n], u*[T,m]) of the affine model.

    Raises ValueError with the reference's message (:139-140) if the Riccati step is not SPD or
    the unconstrained minimiser violates an absolute bound (then the Riccati solution is not the
    QP solution and the comparison is not well-posed — SURVEY.md section 0)."""
    if indices_u_into_x is not None or x_bound_rel is not None or u_bound_rel is not None:
        raise NotImplementedError("out of scope: position-controlled / relative-bound TVLQR")
    T = At.shape[0]
    try:
        K, k = tvlqr_riccati(At, Bt, ct, Q, Qd, R, x_trj_d)
    except np.linalg.LinAlgError:
        raise ValueError("TV_LQR failed. Optimization problem is not solved.")
    n = Q.shape[0]
    m = R.shape[0]
    xs = np.zeros((T + 1, n))
    us = np.zeros((T, m))
    xs[0] = x0
    for t in range(T):
        us[t] = K[t].dot(xs[t]) + k[t]
        xs[t + 1] = At[t].dot(xs[t]) + Bt[t].dot(us[t]) + ct[t]
    if x_bound_abs is not None:
        lo, hi = np.asarray(x_bound_abs[0]), np.asarray(x_bound_abs[1])
        if np.any(xs[1:] < lo[1:T + 1] - bound_tol) or np.any(xs[1:] > hi[1:T + 1] + bound_tol):
            raise ValueError("TV_LQR failed. Optimization problem is not solved.")
    if u_bound_abs is not None:
        lo, hi = np.asarray(u_bound_abs[0]), np.asarray(u_bound_abs[1])
        if np.any(us < lo[:T] - bound_tol) or np.any(us > hi[:T] + bound_tol):
            raise ValueError("TV_LQR failed. Optimization problem is not solved.")
    return xs, us


def closed_loop_descent(system, K, k, x0):
    """irs_lqr/irs_lqr.py:169-184: re-solving the remaining-horizon QP from the actual state and
    applying u*[0] equals applying u_t = K_t x_t + k_t (Bellman), then stepping the TRUE dynamics."""
    T = K.shape[0]
    x_new = np.zeros((T + 1, system.dim_x))
    u_new = np.zeros((T, system.dim_u))
    x_new[0] = x0
    for t in range(T):
        u_new[t] = K[t].dot(x_new[t]) + k[t]
        x_new[t + 1] = system.dynamics(x_new[t], u_new[t])
    return x_new, u_new


class IrsLqrOracle:
    """irs_lqr/irs_lqr.py:34-218 restated (float64): construction, local_descent, iterate.

    mode: "exact" | "first_order" | "zero_order"; `sampling(xbar, ubar, iter) -> (dx, du)` as in
    irs_lqr_zero_order.py:12-22.  Box bounds are not modelled (inactive-bound regime only)."""

    def __init__(self, system, Q, Qd, R, x0, xd_trj, u_trj_initial, mode="exact", sampling=None,
                 verbose=False):
        self.system, self.Q, self.Qd, self.R = system, Q, Qd, R
        self.x0, self.xd_trj = np.asarray(x0, dtype=np.float64), xd_trj
        self.mode, self.sampling, self.verbose = mode, sampling, verbose
        self.u_trj = np.asarray(u_trj_initial, dtype=np.float64)
        self.T = self.u_trj.shape[0]
        self.x_trj = rollout(system, self.x0, self.u_trj)                    # :61
        self.cost = evaluate_cost(self.x_trj, self.u_trj, xd_trj, Q, R)      # :62
        self.x_trj_lst, self.u_trj_lst, self.cost_lst = [self.x_trj], [self.u_trj], [self.cost]
        self.iter = 1                                                        # :71
        self.start_time = time.time()

    def sample_deltas(self, x_trj, u_trj):
        n = self.system.dim_x
        rows = []
        for t in range(self.T):
            dx, du = self.sampling(x_trj[t], u_trj[t], self.iter)
            rows.append(np.hstack((dx, du)))
        return np.stack(rows)

    def get_TV_matrices(self, x_trj, u_trj):
        if self.mode == "exact":
            return exact_tv_matrices(self.system, x_trj, u_trj)
        deltas = self.sample_deltas(x_trj, u_trj)
        if self.mode == "first_order":
            return first_order_tv_matrices(self.system, x_trj, u_trj, deltas)
        return zero_order_tv_matrices(self.system, x_trj, u_trj, deltas)

    def local_descent(self, x_trj, u_trj):
        # :148-186
        At, Bt, ct = self.get_TV_matrices(x_trj, u_trj)
        K, k = tvlqr_riccati(At, Bt, ct, self.Q, self.Qd, self.R, self.xd_trj)
        return closed_loop_descent(self.system, K, k, x_trj[0])

    def iterate(self, max_iterations):
        # :188-218 — runs max_iterations+1 descents; the last one is logged but not adopted.
        while True:
            x_new, u_new = self.local_descent(self.x_trj, self.u_trj)
            cost_new = evaluate_cost(x_new, u_new, self.xd_trj, self.Q, self.R)
            if self.verbose:
                print("Iteration: {:02d} ".format(self.iter) + " || " +
                      "Current Cost: {0:05f} ".format(cost_new))
            self.x_trj_lst.append(x_new)
            self.u_trj_lst.append(u_new)
            self.cost_lst.append(cost_new)
            if self.iter > max_iterations:
                break
            self.cost, self.x_trj, self.u_trj = cost_new, x_new, u_new
            self.iter += 1
        return self.x_trj, self.u_trj, self.cost
