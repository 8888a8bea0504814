"""solve_tvlqr / get_solver with the reference's signatures (irs_lqr/tv_lqr.py:11-145).

The reference builds a Drake MathematicalProgram QP and calls OSQP.  Here the same optimisation
problem is solved by an affine Riccati recursion on the GPU (csrc/tvlqr.cuh) — exact, not
iterative — which is the QP's minimiser whenever no box bound is active.  When an absolute bound
IS active, the QP is solved by ADMM on the box split with Riccati-structured linear solves
(csrc/tvlqr_box.cuh; same algorithm as oracle/box_tvlqr.py, which is checked against a dense QP
solve); the boxes may vary over the horizon as in the reference (x_bound_abs[:, t], u_bound_abs[:, t]).

Relative bounds: the reference bounds the auxiliary variables dxt / dut (tv_lqr.py:119-124), which it
ties to x / u only inside `if indices_u_into_x is not None` (:100-108).  With indices_u_into_x=None —
the analytic-dynamics hot path — they are free variables, so x_bound_rel / u_bound_rel constrain
nothing unless a lower bound exceeds its upper bound (infeasible QP -> the reference's ValueError).
That literal behaviour is reproduced.  The position-controlled variant (indices_u_into_x given) belongs
to the quasistatic drivers and is not implemented.

Start state: the reference also boxes xt[0] = x0 (:113-114), so an x0 outside x_bound_abs[:, 0] makes
the QP infeasible; reproduced (ValueError).  xinit / uinit are initial guesses of an iterative solver;
the solves here are direct (or warm-started internally) and ignore them.
"""
import numpy as np
import torch

from . import _device, _lib

_SOLVER_NAMES = ("osqp", "snopt", "clp", "scs", "gurobi")
TVLQR_FAILED = "TV_LQR failed. Optimization problem is not solved."


class RiccatiSolver:
    """Stand-in for the Drake solver objects returned by the reference's get_solver."""

    def __init__(self, name):
        self.name = name

    def __repr__(self):
        return "RiccatiSolver(requested=%r)" % self.name


def get_solver(solver_name):
    # tv_lqr.py:11-27: unknown names raise ValueError("Do not recognize solver.")
    if solver_name in _SOLVER_NAMES:
        return RiccatiSolver(solver_name)
    raise ValueError("Do not recognize solver.")


def riccati_device(At, Bt, ct, Q, Qd, R, xd, xd_stride):
    """Device-level backward pass.  At [I,T,n,n] ... -> K [I,T,m,n], k [I,T,m], status [I]."""
    I, T, n, _ = At.shape
    m = Bt.shape[3]
    K = _device.empty((I, T, m, n))
    k = _device.empty((I, T, m))
    status = _device.empty((I,), torch.int32)
    _lib.call("irs_tvlqr_riccati", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
              _device.ptr(Q), _device.ptr(Qd), _device.ptr(R), _device.ptr(xd), int(xd_stride),
              I, T, _device.ptr(K), _device.ptr(k), _device.ptr(status), _device.stream_ptr())
    return K, k, status


# ADMM parameters of the bounded solve (csrc/tvlqr_box.cuh)
BOX_RHO0 = 1.0
BOX_ALPHA = 1.6
BOX_EPS = 1e-10
BOX_MAX_ITER = 100000
BOUND_TOL = 1e-9


def box_penalties(Q, R, rho0=BOX_RHO0):
    """Per-coordinate ADMM penalties: rho0 times the cost curvature of the coordinate, floored at the
    mean curvature (a coordinate with zero weight still gets a usable penalty)."""
    qd = np.diag(np.asarray(Q, dtype=np.float64)).copy()
    rd = 0.5 * np.diag(np.asarray(R, dtype=np.float64))
    return rho0 * np.maximum(qd, qd.mean()), rho0 * np.maximum(rd, rd.mean())


def box_solve_device(system, mpc, At, Bt, ct, dQ, dQd, dR, Q, Qd, R, dxd, xd_stride, x0, xlo, xhi, ulo, uhi,
                     K0=None, k0=None, rho0=BOX_RHO0, alpha=BOX_ALPHA, eps=BOX_EPS, max_iter=BOX_MAX_ITER):
    """Bounded solve on the device.  xlo / xhi: [n] (constant box) or [T+1, n] (one box per timestep);
    ulo / uhi: [m] or [T, m].  At [I,T,n,n] ... CUDA float64; Q, Qd, R numpy (for the penalty
    augmentation).  mpc=True: the reference's closed loop on the true dynamics of `system`
    (irs_lqr.py:169-184), K0/k0 = the unconstrained gains (start times whose unconstrained plan stays
    inside the box skip their QP); mpc=False: one QP from x0 (tv_lqr.py:69-145).  Returns device tensors
    (x_trj [I,T+1,n], u_trj [I,T,m], cost [I], status [I], iters [I])."""
    I, T, n, _ = At.shape
    m = Bt.shape[3]
    dx, du = box_penalties(Q, R, rho0)
    Qe = _device.to_device(np.asarray(Q, dtype=np.float64) + 0.5 * np.diag(dx))
    Qde = _device.to_device(np.asarray(Qd, dtype=np.float64) + 0.5 * np.diag(dx))
    Re = _device.to_device(np.asarray(R, dtype=np.float64) + np.diag(du))      # halved inside the kernel
    K = _device.empty((I, T, m, n))
    k = _device.empty((I, T, m))
    Hinv = _device.empty((I, T, m, m))
    P = _device.empty((I, T + 1, n, n))
    rstatus = _device.empty((I,), torch.int32)
    _lib.call("irs_tvlqr_riccati_ex", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
              _device.ptr(Qe), _device.ptr(Qde), _device.ptr(Re), _device.ptr(dxd), int(xd_stride), I, T,
              _device.ptr(K), _device.ptr(k), _device.ptr(rstatus), _device.ptr(Hinv), _device.ptr(P),
              _device.stream_ptr())
    x_trj = _device.empty((I, T + 1, n))
    u_trj = _device.empty((I, T, m))
    cost = _device.empty((I,))
    status = _device.empty((I,), torch.int32)
    iters = _device.empty((I,), torch.int32)
    d = {name: _device.to_device(np.ascontiguousarray(v, dtype=np.float64))
         for name, v in (("dx", dx), ("du", du), ("xlo", xlo), ("xhi", xhi), ("ulo", ulo), ("uhi", uhi))}
    prm, nprm = system._params()
    xbox_stride = n if np.ndim(xlo) == 2 else 0
    ubox_stride = m if np.ndim(ulo) == 2 else 0
    if (xbox_stride and np.shape(xlo) != (T + 1, n)) or (ubox_stride and np.shape(ulo) != (T, m)):
        raise ValueError("time-varying boxes must be [T+1, n] (states) and [T, m] (inputs)")
    _lib.call("irs_tvlqr_box_solve", system.system_id, prm, nprm, 1 if mpc else 0, _device.ptr(At),
              _device.ptr(Bt), _device.ptr(ct), _device.ptr(K), _device.ptr(Hinv), _device.ptr(P),
              _device.ptr(dQ), _device.ptr(dQd), _device.ptr(dR), _device.ptr(dxd), int(xd_stride),
              _device.ptr(d["dx"]), _device.ptr(d["du"]), _device.ptr(d["xlo"]), _device.ptr(d["xhi"]),
              _device.ptr(d["ulo"]), _device.ptr(d["uhi"]), xbox_stride, ubox_stride, _device.ptr(x0),
              _device.ptr(K0), _device.ptr(k0),
              BOUND_TOL, float(alpha), float(eps), int(max_iter), I, T, _device.ptr(x_trj), _device.ptr(u_trj), _device.ptr(cost),
              _device.ptr(status), _device.ptr(iters), _device.stream_ptr())
    return x_trj, u_trj, cost, status | rstatus, iters


class _DimsOnlySystem:
    """solve_tvlqr knows only (n, m): the bounded single-QP solve never evaluates the dynamics, but the
    kernel is instantiated per built-in system; pick the one with matching dimensions."""
    _BY_DIMS = {(2, 1): (0, [0.05]), (5, 2): (1, [0.1]), (12, 4): (2, [0.05, 0.775, 0.15, 9.81, 0.0015, 0.0025,
                                                                      0.0035, 1.0, 0.0245]),
                (6, 2): (3, [0.05, 0.2])}

    def __init__(self, n, m):
        if (n, m) not in self._BY_DIMS:
            raise NotImplementedError("bounded TVLQR is instantiated for the built-in system dimensions only")
        self.system_id, self._p = self._BY_DIMS[(n, m)]

    def _params(self):
        return _lib.params_array(self._p)


def _box_rows(bound, rows, dim, name):
    """The reference indexes its bounds by timestep (x_bound_abs[0, t]: tv_lqr.py:113-116): accepts
    [2, rows, dim] (or [2, dim], broadcast over the horizon) -> (lo, hi), each [dim] when the box is
    constant over the horizon, else [rows, dim]."""
    lo, hi = np.asarray(bound[0], dtype=np.float64), np.asarray(bound[1], dtype=np.float64)
    if lo.ndim == 1:
        lo, hi = np.tile(lo, (rows, 1)), np.tile(hi, (rows, 1))
    if lo.shape[0] < rows or lo.shape[1] != dim or hi.shape != lo.shape:
        raise ValueError("%s must hold %d rows of %d bounds" % (name, rows, dim))
    lo, hi = np.ascontiguousarray(lo[:rows]), np.ascontiguousarray(hi[:rows])
    if np.all(lo == lo[0]) and np.all(hi == hi[0]):
        return lo[0], hi[0]
    return lo, hi


def _violates(v, lo, hi, tol=BOUND_TOL):
    return bool(np.any(v < np.asarray(lo) - tol) or np.any(v > np.asarray(hi) + tol))


def solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, x_trj_d, solver=None, indices_u_into_x=None,
                x_bound_abs=None, u_bound_abs=None, x_bound_rel=None, u_bound_rel=None,
                xinit=None, uinit=None):
    """Same arguments and return value as the reference (tv_lqr.py:30-33, :142-145):
    numpy float64 in, (x*[T+1,n], u*[T,m]) out.  ValueError(TVLQR_FAILED) on failure (:139-140)."""
    if indices_u_into_x is not None:
        raise NotImplementedError(
            "position-controlled TVLQR (indices_u_into_x) belongs to the quasistatic drivers, outside the "
            "analytic-dynamics hot path")
    for rel in (x_bound_rel, u_bound_rel):
        # bounds on the free variables dxt / dut (see the module docstring): inert unless infeasible
        if rel is not None and np.any(np.asarray(rel[0], dtype=np.float64) > np.asarray(rel[1], dtype=np.float64)):
            raise ValueError(TVLQR_FAILED)
    At = np.asarray(At, dtype=np.float64)
    Bt = np.asarray(Bt, dtype=np.float64)
    T, n, m = At.shape[0], At.shape[1], Bt.shape[2]
    ct = np.asarray(ct, dtype=np.float64).reshape(T, n)
    dA = _device.to_device(At[None])
    dB = _device.to_device(Bt[None])
    dc = _device.to_device(ct[None])
    dQ, dQd, dR = _device.to_device(Q), _device.to_device(Qd), _device.to_device(R)
    dxd = _device.to_device(np.asarray(x_trj_d, dtype=np.float64)[:T + 1])
    dx0 = _device.to_device(np.asarray(x0, dtype=np.float64)[None])
    K, k, status = riccati_device(dA, dB, dc, dQ, dQd, dR, dxd, 0)
    xs = _device.empty((1, T + 1, n))
    us = _device.empty((1, T, m))
    _lib.call("irs_tvlqr_linear_rollout", n, m, _device.ptr(dA), _device.ptr(dB), _device.ptr(dc),
              _device.ptr(K), _device.ptr(k), _device.ptr(dx0), 1, T, _device.ptr(xs),
              _device.ptr(us), _device.stream_ptr())
    if int(status.item()) != 0:
        raise ValueError(TVLQR_FAILED)
    xs = _device.to_numpy(xs[0])
    us = _device.to_numpy(us[0])
    if not (np.all(np.isfinite(xs)) and np.all(np.isfinite(us))):
        raise ValueError(TVLQR_FAILED)
    big = 1e30
    xlo, xhi = (_box_rows(x_bound_abs, T + 1, n, "x_bound_abs") if x_bound_abs is not None
                else (-big * np.ones(n), big * np.ones(n)))
    ulo, uhi = (_box_rows(u_bound_abs, T, m, "u_bound_abs") if u_bound_abs is not None
                else (-big * np.ones(m), big * np.ones(m)))
    if np.any(xlo > xhi) or np.any(ulo > uhi):
        raise ValueError(TVLQR_FAILED)                      # empty box: infeasible QP
    # xt[0] = x0 is boxed too (tv_lqr.py:113-114): a start state outside its box is an infeasible QP
    if _violates(xs[0], xlo[0] if xlo.ndim == 2 else xlo, xhi[0] if xhi.ndim == 2 else xhi):
        raise ValueError(TVLQR_FAILED)
    x_active = _violates(xs[1:], xlo[1:] if xlo.ndim == 2 else xlo, xhi[1:] if xhi.ndim == 2 else xhi)
    u_active = _violates(us, ulo, uhi)
    if not (x_active or u_active):
        return xs, us
    # an absolute bound is active: box-constrained QP (tv_lqr.py:113-118, :132-134)
    xb, ub, _, bstatus, _ = box_solve_device(_DimsOnlySystem(n, m), False, dA, dB, dc, dQ, dQd, dR, Q, Qd, R,
                                             dxd, 0, dx0, xlo, xhi, ulo, uhi)
    if int(bstatus.item()) != 0:
        raise ValueError(TVLQR_FAILED)
    return _device.to_numpy(xb[0]), _device.to_numpy(ub[0])
