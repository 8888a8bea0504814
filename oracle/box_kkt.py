"""TEST INFRASTRUCTURE ONLY — an exact optimality certificate for the box-constrained TVLQR QP.

The QP of irs_lqr/tv_lqr.py:69-137 with absolute boxes (:113-118, :132-134):

    minimise   sum_{t<T} (x_t-xd_t)'Q(x_t-xd_t) + 1/2 u_t'R u_t  +  (x_T-xd_T)'Qd(x_T-xd_T)
    s.t.       x_{t+1} = A_t x_t + B_t u_t + c_t,   xlo <= x_t <= xhi (t >= 1),   ulo <= u_t <= uhi

This module shares nothing with the ADMM (oracle/box_tvlqr.py) nor with the Riccati recursion.  The states
are condensed out (x = s0 + Su u, x_0 fixed), the weights enter as in oracle/dense_lqr.py (gradient of
(x-d)'W(x-d) is (W + W')(x - d)), and the boxes become rows of G u <= h.  `certify` takes the active set
from a candidate, solves the equality-constrained KKT system on that set in float64 and checks the two
conditions that make the result the global minimiser of a convex QP: multipliers >= 0 and no violated
inactive row (and a KKT system that the solve really satisfied: rows of the set may be dependent).  `bvls`
is a second, solver-based reference for input-only boxes.
"""
import numpy as np


def _sym(W):
    W = np.asarray(W, dtype=np.float64)
    return 0.5 * (W + W.T)


def _rows(b, T, first):
    """A box given as [dim] (constant) or [rows, dim] (one per timestep) -> [T, dim] for steps first..first+T-1."""
    b = np.asarray(b, dtype=np.float64)
    return np.tile(b, (T, 1)) if b.ndim == 1 else b[first:first + T]


class BoxQP:
    def __init__(self, At, Bt, ct, Q, Qd, R, x0, xd, xlo, xhi, ulo, uhi):
        At, Bt, ct = (np.asarray(v, dtype=np.float64) for v in (At, Bt, ct))
        T, n, m = At.shape[0], At.shape[1], Bt.shape[2]
        self.T, self.n, self.m = T, n, m
        x0 = np.asarray(x0, dtype=np.float64)
        xd = np.asarray(xd, dtype=np.float64)[:T + 1]
        # x_{1..T} = s0 + Su u
        Su = np.zeros((T * n, T * m))
        s0 = np.zeros(T * n)
        prev_s, prev_S = x0, np.zeros((n, T * m))
        for t in range(T):
            S = At[t].dot(prev_S)
            S[:, t * m:(t + 1) * m] += Bt[t]
            s = At[t].dot(prev_s) + ct[t]
            Su[t * n:(t + 1) * n], s0[t * n:(t + 1) * n] = S, s
            prev_s, prev_S = s, S
        self.Su, self.s0, self.x0 = Su, s0, x0
        # Hessian blocks W + W' of x_1..x_T (Qd for x_T), sym(R) of every u; gradient offset -(W + W') xd
        W2 = np.zeros((T, n, n))
        W2[:] = 2.0 * _sym(Q)
        W2[T - 1] = 2.0 * _sym(Qd)
        self.W2 = W2
        self.e0 = e0 = (s0 - xd[1:].reshape(-1)).reshape(T, n)
        We0 = np.einsum("tij,tj->ti", W2, e0).reshape(-1)
        WS = np.einsum("tij,tjk->tik", W2, Su.reshape(T, n, T * m)).reshape(T * n, T * m)
        self.H = Su.T.dot(WS) + np.kron(np.eye(T), _sym(R))
        self.H = 0.5 * (self.H + self.H.T)
        self.g = Su.T.dot(We0)
        # G u <= h: x upper, x lower, u upper, u lower (rows with an infinite bound are left out)
        xl, xh = _rows(xlo, T, 1).reshape(-1), _rows(xhi, T, 1).reshape(-1)
        ul, uh = _rows(ulo, T, 0).reshape(-1), _rows(uhi, T, 0).reshape(-1)
        Iu = np.eye(T * m)
        G = np.vstack((Su, -Su, Iu, -Iu))
        h = np.concatenate((xh - s0, s0 - xl, uh, -ul))
        keep = np.isfinite(h)
        self.G, self.h = G[keep], h[keep]
        # the bound value of each row, for a scale of its slack
        self.bound = np.concatenate((xh, xl, uh, ul))[keep]

    def states(self, u):
        """[T+1, n] rollout of u [T, m] through the affine model."""
        xs = self.s0 + self.Su.dot(np.asarray(u, dtype=np.float64).reshape(-1))
        return np.vstack((self.x0[None], xs.reshape(self.T, self.n)))

    def objective(self, u):
        uv = np.asarray(u).reshape(-1)
        return 0.5 * uv.dot(self.H).dot(uv) + self.g.dot(uv)

    def kkt(self, active):
        """Minimiser with the rows `active` held as equalities -> (u [T m], multipliers [len(active)])."""
        A = np.flatnonzero(active)
        N, k = self.H.shape[0], A.size
        M = np.zeros((N + k, N + k))
        M[:N, :N] = self.H
        M[:N, N:] = self.G[A].T
        M[N:, :N] = self.G[A]
        rhs = np.concatenate((-self.g, self.h[A]))
        try:
            z = np.linalg.solve(M, rhs)
        except np.linalg.LinAlgError:           # dependent rows: no unique point; the residual test rejects it
            z = np.linalg.lstsq(M, rhs, rcond=None)[0]
        return z[:N], z[N:]

    def slack(self, u):
        return self.h - self.G.dot(np.asarray(u).reshape(-1))

    def certify(self, u_candidate, delta=1e-6, tol=1e-9):
        """Active set of the candidate (rows with slack <= delta max(1, |bound|)), the exact minimiser on it
        and the two optimality conditions.  Returns a dict: x, u (exact), lam (one per row, 0 off the active
        set), active, min_lam (relative to the largest multiplier), max_violation (of the inactive rows,
        relative to max(1, |bound|)) and certified."""
        scale = np.maximum(1.0, np.abs(self.bound))
        active = self.slack(u_candidate) <= delta * scale
        return self.at(active, tol)

    def at(self, active, tol=1e-9):
        """The exact minimiser with the rows `active` held as equalities and its optimality conditions (the
        dict of `certify`)."""
        u, lam_a = self.kkt(active)
        lam = np.zeros(self.h.size)
        lam[active] = lam_a
        scale = np.maximum(1.0, np.abs(self.bound))
        lam_scale = max(float(np.max(np.abs(lam))), 1e-300)
        viol = -self.slack(u) / scale
        max_violation = float(np.max(viol[~active])) if np.any(~active) else -np.inf
        min_lam = float(np.min(lam_a)) / lam_scale if lam_a.size else np.inf
        # stationarity and the active rows, relative to the size of their terms
        Ga = self.G[active]
        stat = self.H.dot(u) + self.g + Ga.T.dot(lam_a)
        stat_scale = float(np.max(np.abs(self.H).dot(np.abs(u)) + np.abs(self.g) + np.abs(Ga.T).dot(np.abs(lam_a))))
        kkt_residual = max(float(np.max(np.abs(stat))) / max(stat_scale, 1e-300),
                           float(np.max(np.abs(Ga.dot(u) - self.h[active]) / scale[active], initial=0.0)))
        return dict(u=u.reshape(self.T, self.m), x=self.states(u), lam=lam, active=active, min_lam=min_lam,
                    max_violation=max_violation, kkt_residual=kkt_residual,
                    certified=bool(min_lam >= -tol and max_violation <= tol and kkt_residual <= 1e-9))

    def margins(self, r):
        """Strict complementarity of a solution: (smallest active multiplier relative to the largest, smallest
        inactive slack relative to max(1, |bound|))."""
        scale = np.maximum(1.0, np.abs(self.bound))
        lam_a = r["lam"][r["active"]]
        lam_rel = float(np.min(lam_a)) / max(float(np.max(np.abs(r["lam"]))), 1e-300) if lam_a.size else np.inf
        s = self.slack(r["u"].reshape(-1)) / scale
        slack_rel = float(np.min(s[~r["active"]])) if np.any(~r["active"]) else np.inf
        return lam_rel, slack_rel


def bvls(qp, Q, Qd, R, ulo, uhi):
    """Input boxes only: the cost written as a bounded linear least-squares problem and solved by scipy's BVLS,
    without the condensed Hessian: with sym(W) = L L', (x-d)'W(x-d) = |L'(x-d)|^2 and 1/2 u'Ru = |L_R' u|^2 / 2,
    so the residual stacks L_t'(s0 + Su u - xd)_t over t and L_R' u / sqrt(2) over the inputs."""
    from scipy.optimize import lsq_linear
    T, n, m = qp.T, qp.n, qp.m
    Lq, Lqd, Lr = (np.linalg.cholesky(_sym(W)) for W in (Q, Qd, R))
    Lx = [Lqd.T if t == T - 1 else Lq.T for t in range(T)]
    Fx = np.zeros((T * n, T * n))
    for t in range(T):
        Fx[t * n:(t + 1) * n, t * n:(t + 1) * n] = Lx[t]
    A = np.vstack((Fx.dot(qp.Su), np.kron(np.eye(T), Lr.T / np.sqrt(2.0))))
    b = np.concatenate((-Fx.dot(qp.e0.reshape(-1)), np.zeros(T * m)))
    lo, hi = _rows(ulo, T, 0).reshape(-1), _rows(uhi, T, 0).reshape(-1)
    res = lsq_linear(A, b, bounds=(lo, hi), method="bvls", tol=1e-15, max_iter=10000)
    return res.x.reshape(T, m), res


# ------------------------------------------------------------------------------------------------
# well-posed test problems
# ------------------------------------------------------------------------------------------------
BIG = 1e30          # "no bound" (what solve_tvlqr passes for an absent box)


def _spd(rng, d, lo=0.5):
    M = rng.standard_normal((d, d))
    return M.dot(M.T) / d + lo * np.eye(d)


def weights(rng, n, m, kind):
    """(Q, Qd, R) of a kind: diag, dense (SPD) or nonsym (SPD symmetric parts plus skew parts)."""
    if kind == "diag":
        return np.diag(rng.uniform(0.5, 2, n)), np.diag(rng.uniform(5, 20, n)), np.diag(rng.uniform(0.5, 2, m))
    Q, Qd, R = _spd(rng, n), 10 * _spd(rng, n), _spd(rng, m)
    if kind == "nonsym":
        Q, Qd, R = (W + (lambda S: S - S.T)(rng.standard_normal(W.shape)) for W in (Q, Qd, R))
    return Q, Qd, R


def make_problem(n, m, T, box, kind="dense", I=1, inactive=(), shared_xd=False, seed=0):
    """I instances of a random problem with stable dynamics (||A_t||_2 = 0.95, so long horizons stay bounded)
    and one box shared by all instances, as the kernel takes it.

    box: "input" (every input, both sides), "state" (half the state coordinates, both sides), "both",
         "tv" (both, one box per timestep: xlo/xhi [T+1, n], ulo/uhi [T, m]) or "wide" (1e4: nothing active).
    The box is symmetric about 0, its half-width the 70th percentile of |value| over the unconstrained
    minimisers of the active instances (85th / 95th for states / inputs when both are boxed), so that
    several rows on both sides are active.  Instances listed in
    `inactive` get x0, xd and c_t a hundred times smaller: their minimiser stays deep inside the box.
    Returns a dict of numpy arrays (At [I,T,n,n] ... , xd [I or 1, T+1, n], x0 [I,n], Q, Qd, R, xlo, xhi,
    ulo, uhi)."""
    rng = np.random.default_rng(seed)
    M = np.eye(n) + 0.3 * rng.standard_normal((I, T, n, n))
    At = 0.95 * M / np.linalg.norm(M, ord=2, axis=(2, 3))[..., None, None]
    Bt = 0.5 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    xd = rng.standard_normal((1 if shared_xd else I, T + 1, n))
    x0 = rng.standard_normal((I, n))
    Q, Qd, R = weights(rng, n, m, kind)
    if shared_xd and inactive:
        raise ValueError("inactive instances need their own xd")
    for i in inactive:
        x0[i] *= 0.01
        xd[i] *= 0.01
        ct[i] *= 0.01
    act = [i for i in range(I) if i not in inactive]
    free = []
    for i in act:
        qp = BoxQP(At[i], Bt[i], ct[i], Q, Qd, R, x0[i], xd[0 if shared_xd else i], np.full(n, np.inf),
                   np.full(n, np.inf), np.full(m, np.inf), np.full(m, np.inf))
        uf = np.linalg.solve(qp.H, -qp.g)
        free.append((qp.states(uf)[1:], uf.reshape(T, m)))
    xs, us = np.stack([f[0] for f in free]), np.stack([f[1] for f in free])
    # with both boxes the state box is looser and the input box looser still, so that the inputs can hold it
    both = box in ("both", "tv")
    xa = np.quantile(np.abs(xs).reshape(-1, n), 0.85 if both else 0.7, axis=0)
    ua = np.quantile(np.abs(us).reshape(-1, m), 0.95 if both else 0.7, axis=0)
    xhi, uhi = np.full(n, BIG), np.full(m, BIG)
    if box in ("input", "both", "tv"):
        uhi = ua
    if box in ("state", "both", "tv"):
        coords = rng.permutation(n)[:max(1, n // 2)]
        xhi[coords] = xa[coords]
    if box == "wide":
        xhi, uhi = np.full(n, 1e4), np.full(m, 1e4)
    p = dict(At=At, Bt=Bt, ct=ct, xd=xd, x0=x0, Q=Q, Qd=Qd, R=R, n=n, m=m, T=T, I=I, shared_xd=shared_xd)
    for _ in range(20):
        xlo_, xhi_, ulo_, uhi_ = _breathe(box, T, xhi, uhi)
        p.update(xlo=xlo_, xhi=xhi_, ulo=ulo_, uhi=uhi_)
        # feasible with room to spare: the state box shrunk by a fifth still admits inputs inside theirs
        # (a box that is only just feasible leaves the ADMM a feasible set without interior)
        p.update(xlo=np.where(xlo_ > -BIG, 0.8 * xlo_, xlo_), xhi=np.where(xhi_ < BIG, 0.8 * xhi_, xhi_))
        room = all(feasible(instance_qp(p, i)) for i in act)
        p.update(xlo=xlo_, xhi=xhi_)
        if room:
            return p
        xhi = np.where(xhi < BIG, 1.25 * xhi, BIG)    # the inputs cannot hold the state box: widen it
    raise RuntimeError("no feasible box")


def _breathe(box, T, xhi, uhi):
    if box == "tv":
        # a box that breathes over the horizon: +-20 % of its half-width
        wave_x = 1.0 + 0.2 * np.sin(0.7 * np.arange(T + 1))[:, None]
        wave_u = 1.0 + 0.2 * np.cos(0.5 * np.arange(T))[:, None]
        xhi = np.where(xhi < BIG, xhi * wave_x, BIG)
        uhi = uhi * wave_u
    return -xhi, xhi, -uhi, uhi


def feasible(qp):
    """Is there an input sequence inside the input box that keeps the states inside theirs?  (An LP.)"""
    from scipy.optimize import linprog
    N = qp.T * qp.m
    xrows = np.flatnonzero(np.abs(qp.bound[:qp.h.size - 2 * N]) < BIG)
    lo, hi = -qp.h[qp.h.size - N:], qp.h[qp.h.size - 2 * N:qp.h.size - N]
    if xrows.size == 0:
        return True
    res = linprog(np.zeros(N), A_ub=qp.G[xrows], b_ub=qp.h[xrows], bounds=list(zip(lo, hi)), method="highs")
    return res.status == 0


def instance_qp(p, i, scale=1.0):
    """BoxQP of instance i of make_problem's dict (weights times `scale`: the same minimiser)."""
    return BoxQP(p["At"][i], p["Bt"][i], p["ct"][i], scale * p["Q"], scale * p["Qd"], scale * p["R"], p["x0"][i],
                 p["xd"][0 if p["shared_xd"] else i], p["xlo"], p["xhi"], p["ulo"], p["uhi"])
