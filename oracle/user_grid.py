"""TEST INFRASTRUCTURE ONLY — a user-written system of any (N, M) and its float64 twin.

One step body and one Jacobian body (CUDA C++, for user_system.CudaSourceDynamics) that compile for every
N + M <= 16 and touch every state and input with a coefficient of its own, so that a transposed or misplaced
Gram entry, or N and M swapped somewhere, changes the numbers:

    f_i = p0 x_i + h (sin x_{(i+1)%N} + p1 x_{(i+2)%N} u_{i%M} + sum_k c_ik u_k),
    c_ik = (1 + (3i + k) mod 5) / 4 * (-1)^(i+k)

with p = PARAMS = [0.9, 0.3, 0.7] (p2 unused: it only makes IRS_USER_NPARAMS differ from the used count).
p0 < 1 makes the map mildly contractive, so long rollouts stay well-conditioned.  The Jacobian body
accumulates with +=, so the coinciding indices of N <= 2 add up.

`GridOracle(n, m, h)` has the interface oracle/cpu_restatement.py expects (dim_x, dim_u, h, dynamics,
dynamics_batch, jacobian_xu, jacobian_xu_batch), so cr.rollout, cr.evaluate_cost, cr.affine_offset,
oracle/box_tvlqr.py and oracle/box_kkt.py take it unchanged.
"""
import numpy as np

PARAMS = [0.9, 0.3, 0.7]
H = 0.05

_COEFF = "R((1 + (3 * i + k) % 5)) * R(0.25) * R(((i + k) & 1) ? -1 : 1)"


def step_source():
    return """
    for (int i = 0; i < N; ++i) {
        R s, c;
        Math<R>::sincos(x[(i + 1) %% N], s, c);
        R acc = s + p[1] * x[(i + 2) %% N] * u[i %% M];
        for (int k = 0; k < M; ++k) acc += %s * u[k];
        o[i] = p[0] * x[i] + h * acc;
    }
""" % _COEFF


def jacobian_source():
    return """
    for (int e = 0; e < N * D; ++e) J[e] = R(0);
    for (int i = 0; i < N; ++i) {
        R s, c;
        Math<R>::sincos(x[(i + 1) %% N], s, c);
        J[i * D + i] += p[0];
        J[i * D + (i + 1) %% N] += h * c;
        J[i * D + (i + 2) %% N] += h * p[1] * u[i %% M];
        J[i * D + N + i %% M] += h * p[1] * x[(i + 2) %% N];
        for (int k = 0; k < M; ++k) J[i * D + N + k] += h * (%s);
    }
""" % _COEFF


def coeffs(n, m):
    """c [n, m] of the input term."""
    i, k = np.meshgrid(np.arange(n), np.arange(m), indexing="ij")
    return (1 + (3 * i + k) % 5) / 4.0 * np.where((i + k) % 2, -1.0, 1.0)


class GridOracle:
    def __init__(self, n, m, h=H, params=PARAMS):
        self.dim_x, self.dim_u, self.h = n, m, h
        self.p = [float(v) for v in params]
        self.c = coeffs(n, m)
        self.i1 = (np.arange(n) + 1) % n
        self.i2 = (np.arange(n) + 2) % n
        self.im = np.arange(n) % m

    def dynamics_batch(self, x, u):
        x, u = np.atleast_2d(np.asarray(x, dtype=np.float64)), np.atleast_2d(np.asarray(u, dtype=np.float64))
        acc = np.sin(x[:, self.i1]) + self.p[1] * x[:, self.i2] * u[:, self.im] + u @ self.c.T
        return self.p[0] * x + self.h * acc

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]

    def jacobian_xu_batch(self, x, u):
        x, u = np.atleast_2d(np.asarray(x, dtype=np.float64)), np.atleast_2d(np.asarray(u, dtype=np.float64))
        n, h, p = self.dim_x, self.h, self.p
        B = x.shape[0]
        J = np.zeros((B, n, n + self.dim_u))
        J[:, :, n:] += h * self.c[None]
        rows = np.arange(n)
        # np.add.at: the indices coincide for n <= 2 and must add up, as the += of the body
        np.add.at(J, (slice(None), rows, rows), p[0])
        np.add.at(J, (slice(None), rows, self.i1), h * np.cos(x[:, self.i1]))
        np.add.at(J, (slice(None), rows, self.i2), h * p[1] * u[:, self.im])
        np.add.at(J, (slice(None), rows, n + self.im), h * p[1] * x[:, self.i2])
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(x, u)[0]
