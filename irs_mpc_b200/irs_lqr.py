"""IrsLqrParameters / IrsLqr / IrsLqrExact / IrsLqrFirstOrder / IrsLqrZeroOrder.

Same names, constructor signatures, public methods and public state as the reference
(irs_lqr/irs_lqr.py:7-218, irs_lqr_exact.py, irs_lqr_first_order.py, irs_lqr_zero_order.py); the
arithmetic runs in the sm_100a kernels of libirs_mpc_b200.so.  numpy float64 at the API edge.

Differences a user can observe, all deliberate:
  * `local_descent` performs ONE Riccati backward pass + closed-loop rollout instead of T QP
    solves and then verifies, for every start time in parallel, that no planned trajectory touches
    `xbound`/`ubound` — in which case it IS the result of the reference's T QPs (SURVEY.md section 0).
    Otherwise it runs the reference's loop itself with a box-constrained QP at every timestep
    (ADMM with Riccati-structured solves, csrc/tvlqr_box.cuh) — there is no silent clamping.
  * `sampling` may be a `GaussianSampling` object: the noise is then generated inside the kernel.
    Any other callable is honoured through the replay path.
  * only systems derived from `CudaDynamicalSystem` are accepted (no CPU fallback).
"""
import ctypes
import os
import time

import numpy as np
import torch

from . import _device, _lib, smoothing
from ._graph import GraphRunner
from .dynamical_system import CudaDynamicalSystem
from .sampling import GaussianSampling
from .tv_lqr import BOUND_TOL, TVLQR_FAILED, box_solve_device, get_solver, riccati_device


_USE_PIPELINE = os.environ.get("IRS_PIPELINE", "1") != "0"     # see _SampledIrsLqr._pipeline_segments
_PIPELINE_MIN_STEPS = 8                                        # timesteps per segment below which it does not pay
_PIPELINE_SEGMENTS = int(os.environ.get("IRS_PIPELINE_SEGMENTS", "0"))      # 0 = sized from the work per launch
START_BOUND_TOL = 1e-6      # tolerance of the start-state box test in local_descent


class IrsLqrParameters:
    """Attribute bag, irs_lqr/irs_lqr.py:7-31."""

    def __init__(self):
        self.Q = None
        self.Qd = None
        self.R = None
        self.x0 = None
        self.xd_trj = None
        self.u_trj_initial = None
        self.xbound = None
        self.ubound = None
        self.solver_name = "osqp"


class IrsLqr:
    def __init__(self, system, params):
        self.system = system
        self.params = params
        self.check_valid_system(self.system)
        self.check_valid_params(self.params, self.system)

        self.Q = params.Q
        self.Qd = params.Qd
        self.R = params.R
        self.x0 = params.x0
        self.xd_trj = params.xd_trj
        self.u_trj = params.u_trj_initial
        self.xbound = params.xbound
        self.ubound = params.ubound
        self.solver = get_solver(params.solver_name)

        self.T = self.u_trj.shape[0]
        self.dim_x = self.system.dim_x
        self.dim_u = self.system.dim_u

        # device-resident problem data (float64)
        self._dQ = _device.to_device(np.asarray(self.Q, dtype=np.float64))
        self._dQd = _device.to_device(np.asarray(self.Qd, dtype=np.float64))
        self._dR = _device.to_device(np.asarray(self.R, dtype=np.float64))
        self._dxd = _device.to_device(np.asarray(self.xd_trj, dtype=np.float64)[:self.T + 1])
        self._ws = None
        self._db = None
        self._graphs = GraphRunner(system.lib)
        self._last_descent = None

        self.x_trj = self.rollout(self.x0, self.u_trj)
        self.cost = self.evaluate_cost(self.x_trj, self.u_trj)

        self.x_trj_lst = [self.x_trj]
        self.u_trj_lst = [self.u_trj]
        self.cost_lst = [self.cost]

        self.start_time = time.time()
        self.iter = 1

    # -- validation (irs_lqr.py:73-103, same messages) ---------------------------------------
    def check_valid_system(self, system):
        if system.dim_x == 0:
            raise RuntimeError("System has zero states. Did you forget to set dim_x?")
        elif system.dim_u == 0:
            raise RuntimeError("System has zero inputs. Did you forget to set dim_u?")
        if not isinstance(system, CudaDynamicalSystem):
            raise RuntimeError(
                "Could not evaluate dynamics. irs_mpc_b200 runs the dynamics as CUDA functors: the "
                "system must derive from CudaDynamicalSystem (pendulum, bicycle, quadrotor, "
                "three_cart, or your own dynamics as CUDA C++ source in CudaSourceDynamics); there is "
                "no CPU fallback for arbitrary Python dynamics.")
        try:
            system.dynamics(np.zeros(system.dim_x), np.zeros(system.dim_u))
        except _lib.IrsCudaError:
            raise
        except Exception:
            raise RuntimeError("Could not evaluate dynamics. Have you implemented it?")

    def check_valid_params(self, params, system):
        if np.asarray(params.Q).shape != (system.dim_x, system.dim_x):
            raise RuntimeError("Q matrix must be diagonal with dim_x x dim_x.")
        if np.asarray(params.Qd).shape != (system.dim_x, system.dim_x):
            raise RuntimeError("Qd matrix must be diagonal with dim_x x dim_x.")
        if np.asarray(params.R).shape != (system.dim_u, system.dim_u):
            raise RuntimeError("R matrix must be diagonal with dim_u x dim_u.")

    # -- rollout / cost (irs_lqr.py:105-137) ---------------------------------------------------
    def rollout(self, x0, u_trj):
        u = _device.to_device(np.asarray(u_trj, dtype=np.float64).reshape(1, self.T, self.dim_u))
        x0d = _device.to_device(np.asarray(x0, dtype=np.float64).reshape(1, self.dim_x))
        x_trj = _device.empty((1, self.T + 1, self.dim_x))
        cost = _device.empty((1,))
        prm, nprm = self.system._params()
        self.system.lib.call("irs_rollout_open_loop", self.system.system_id, prm, nprm, _device.ptr(u),
                  _device.ptr(x0d), _device.ptr(self._dxd), 0, _device.ptr(self._dQ),
                  _device.ptr(self._dR), 1, self.T, _device.ptr(x_trj), _device.ptr(cost),
                  _device.stream_ptr())
        return _device.to_numpy(x_trj[0])

    def evaluate_cost(self, x_trj, u_trj):
        ld = self._last_descent
        if ld is not None and x_trj is ld[0] and u_trj is ld[1] and np.array_equal(x_trj, ld[2]) \
                and np.array_equal(u_trj, ld[3]):
            # the trajectory local_descent just returned (unmodified): its cost was computed on the
            # device by the same routine (warp_trajectory_cost) during the rollout
            return self._last_descent_cost
        x = _device.to_device(np.asarray(x_trj, dtype=np.float64).reshape(1, self.T + 1, self.dim_x))
        u = _device.to_device(np.asarray(u_trj, dtype=np.float64).reshape(1, self.T, self.dim_u))
        cost = _device.empty((1,))
        self.system.lib.call("irs_evaluate_cost", self.dim_x, self.dim_u, _device.ptr(x), _device.ptr(u),
                  _device.ptr(self._dxd), 0, _device.ptr(self._dQ), _device.ptr(self._dR), 1, self.T,
                  _device.ptr(cost), _device.stream_ptr())
        return float(cost.item())

    # -- linearization -------------------------------------------------------------------------
    def _tv_matrices_device(self, x_nom, u_nom):
        """x_nom [T,n], u_nom [T,m] CUDA float64 -> (At, Bt, ct, status) CUDA tensors."""
        raise NotImplementedError("This class is virtual.")

    def get_TV_matrices(self, x_trj, u_trj):
        """(At[T,n,n], Bt[T,n,m], ct[T,n]) numpy float64, as in the reference."""
        x_nom = _device.to_device(np.asarray(x_trj, dtype=np.float64)[:self.T])
        u_nom = _device.to_device(np.asarray(u_trj, dtype=np.float64)[:self.T])
        At, Bt, ct, status = self._tv_matrices_device(x_nom, u_nom)
        smoothing.check_status(status)
        return _device.to_numpy(At), _device.to_numpy(Bt), _device.to_numpy(ct)

    def _io_bytes(self):
        """(host->device, device->host) bytes one get_TV_matrices call moves."""
        n, m, T = self.dim_x, self.dim_u, self.T
        return T * (n + m) * 8, T * (n * n + n * m + n) * 8 + T * 4

    # -- descent (irs_lqr.py:148-186) ------------------------------------------------------------
    def _descent_buffers(self):
        """Device + pinned host staging for one descent: a single H2D copy of [x_trj | u_trj] and a
        single D2H copy of [x_new | u_new | cost | riccati status | smoothing status]."""
        if self._db is None:
            T, n, m = self.T, self.dim_x, self.dim_u
            db = {}
            nx, nu = (T + 1) * n, T * m
            db["in_dev"] = _device.empty((nx + nu,))
            db["in_host"] = torch.empty((nx + nu,), dtype=torch.float64).pin_memory()
            n_out = nx + nu + 1 + 1 + 1 + (T + 1) // 2
            db["out_dev"] = _device.empty((n_out,))
            db["out_host"] = torch.empty((n_out,), dtype=torch.float64).pin_memory()
            o = db["out_dev"]
            db["x_new"] = o[:nx].view(1, T + 1, n)
            db["u_new"] = o[nx:nx + nu].view(1, T, m)
            db["cost"] = o[nx + nu:nx + nu + 1]
            db["rstatus"] = o[nx + nu + 1:nx + nu + 2].view(torch.int32)[:1]
            db["violated"] = o[nx + nu + 2:nx + nu + 3].view(torch.int32)[:1]
            db["sstatus"] = o[nx + nu + 3:].view(torch.int32)[:T]
            if self.xbound is not None or self.ubound is not None:
                big = 1e30
                xlo, xhi = ((np.asarray(self.xbound[0], dtype=np.float64), np.asarray(self.xbound[1], dtype=np.float64))
                            if self.xbound is not None else (-big * np.ones(n), big * np.ones(n)))
                ulo, uhi = ((np.asarray(self.ubound[0], dtype=np.float64), np.asarray(self.ubound[1], dtype=np.float64))
                            if self.ubound is not None else (-big * np.ones(m), big * np.ones(m)))
                db["box_host"] = (xlo, xhi, ulo, uhi)
                db["box"] = tuple(_device.to_device(np.ascontiguousarray(v)) for v in (xlo, xhi, ulo, uhi))
                db["plan_scratch"] = _device.empty((T * (n + m) * (n + 1),))
            else:
                db["box"] = None
            db["K"] = _device.empty((1, T, m, n))
            db["k"] = _device.empty((1, T, m))
            db["nx"], db["nu"] = nx, nu
            self._db = db
        return self._db

    def _enqueue_descent(self, db):
        """All device work of one descent on the current stream, bracketed by the two staging copies;
        no host synchronisation (this is the sequence the CUDA graph captures)."""
        T, n, m = self.T, self.dim_x, self.dim_u
        nx = db["nx"]
        db["in_dev"].copy_(db["in_host"], non_blocking=True)
        x_all = db["in_dev"][:nx].view(T + 1, n)
        u_nom = db["in_dev"][nx:].view(T, m)
        x_nom = x_all[:T]
        K, k = db["K"], db["k"]
        At, Bt, ct, status = self._linearize_and_riccati(db, x_nom, u_nom)
        db["sstatus"].copy_(status)
        prm, nprm = self.system._params()
        rows_done = None
        if db["box"] is not None:
            # closed-loop rows of the plan check: they need the gains only, so they are computed on a
            # second stream BESIDE the sequential rollout (plain event dependencies: capturable)
            if "plan_stream" not in db:
                db["plan_stream"] = torch.cuda.Stream()
            main, side = torch.cuda.current_stream(), db["plan_stream"]
            gains = torch.cuda.Event()
            gains.record(main)
            side.wait_event(gains)
            with torch.cuda.stream(side):
                self.system.lib.call("irs_tvlqr_plan_rows", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                          _device.ptr(K), _device.ptr(k), 1, T, _device.ptr(db["plan_scratch"]),
                          _device.stream_ptr())
                rows_done = torch.cuda.Event()
                rows_done.record(side)
        self.system.lib.call("irs_rollout_closed_loop", self.system.system_id, prm, nprm, _device.ptr(K),
                  _device.ptr(k), _device.ptr(x_all), _device.ptr(self._dxd), 0,
                  _device.ptr(self._dQ), _device.ptr(self._dR), 1, T, _device.ptr(db["x_new"]),
                  _device.ptr(db["u_new"]), _device.ptr(db["cost"]), _device.stream_ptr())
        if db["box"] is not None:
            # would any of the reference's T re-solved QPs (irs_lqr.py:169-182) have had an active bound?
            xlo, xhi, ulo, uhi = db["box"]
            torch.cuda.current_stream().wait_event(rows_done)
            self.system.lib.call("irs_tvlqr_plan_check", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                      _device.ptr(K), _device.ptr(k), _device.ptr(db["x_new"]), _device.ptr(xlo),
                      _device.ptr(xhi), _device.ptr(ulo), _device.ptr(uhi), BOUND_TOL, 1, T, 1,
                      _device.ptr(db["violated"]), _device.ptr(db["plan_scratch"]), _device.stream_ptr())
        else:
            db["violated"].zero_()
        db["lin"] = (At, Bt, ct)
        db["out_host"].copy_(db["out_dev"], non_blocking=True)

    def _linearize_and_riccati(self, db, x_nom, u_nom):
        """Linearization along the nominal trajectory, then the backward pass -> db["K"], db["k"]."""
        T, n, m = self.T, self.dim_x, self.dim_u
        At, Bt, ct, status = self._tv_matrices_device(x_nom, u_nom)
        self.system.lib.call("irs_tvlqr_riccati", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                  _device.ptr(self._dQ), _device.ptr(self._dQd), _device.ptr(self._dR),
                  _device.ptr(self._dxd), 0, 1, T, _device.ptr(db["K"]), _device.ptr(db["k"]),
                  _device.ptr(db["rstatus"]), _device.stream_ptr())
        return At, Bt, ct, status

    def _graph_key(self):
        """None when this call sequence cannot be replayed from a CUDA graph (see _SampledIrsLqr)."""
        return None

    def _graph_update(self, graph):
        pass

    def _run(self, name, enqueue):
        """Run `enqueue()` eagerly, or — from the third call of the same shape on — replay it from a
        CUDA graph captured through the library (one launch instead of ~8 API calls)."""
        self._graphs.run(name, self._graph_key(), enqueue, self._graph_update)

    def local_descent(self, x_trj, u_trj):
        T, n, m = self.T, self.dim_x, self.dim_u
        db = self._descent_buffers()
        nx, nu = db["nx"], db["nu"]
        if "in_np" not in db:      # numpy views of the pinned mirrors, and the host copy of the box, made once
            db["in_np"], db["out_np"] = db["in_host"].numpy(), db["out_host"].numpy()
            db["sstat_np"] = db["out_np"][nx + nu + 3:].view(np.int32)[:T]
            db["flags_np"] = db["out_np"][nx + nu + 1:nx + nu + 3].view(np.int32)      # [riccati status, ., violated, .]
            if self.xbound is not None:
                db["xbox_np"] = (np.asarray(self.xbound[0], dtype=np.float64) - START_BOUND_TOL,
                                 np.asarray(self.xbound[1], dtype=np.float64) + START_BOUND_TOL)
        h = db["in_np"]
        h[:nx] = np.asarray(x_trj, dtype=np.float64)[:T + 1].reshape(-1)
        h[nx:] = np.asarray(u_trj, dtype=np.float64)[:T].reshape(-1)
        self._run("descent", lambda: self._enqueue_descent(db))
        # one synchronising read-back for everything the host needs
        torch.cuda.current_stream().synchronize()
        o = db["out_np"]
        smoothing.check_status(db["sstat_np"])
        if int(db["flags_np"][0]) != 0:
            raise ValueError(TVLQR_FAILED)
        if int(db["flags_np"][2]) != 0:
            # some planned trajectory touches a bound: the reference's loop with the bounded QP
            x_out, u_out, cost = self._bounded_descent(db)
            finite = np.all(np.isfinite(x_out)) and np.all(np.isfinite(u_out))
        else:
            x_out = o[:nx].reshape(T + 1, n).copy()
            u_out = o[nx:nx + nu].reshape(T, m).copy()
            cost = float(o[nx + nu])
            # the device cost sums every state and input of the trajectory: it is finite iff they all are
            finite = np.isfinite(cost)
        if not finite:
            raise ValueError(TVLQR_FAILED)
        if self.xbound is not None:
            # every QP of the reference's loop also boxes its START state xt[0] = the actual x_t
            # (tv_lqr.py:113-114 at t = 0, called from irs_lqr.py:170-182): a closed-loop state the true
            # dynamics pushed outside xbound makes that QP infeasible -> the reference's ValueError.
            # START_BOUND_TOL: a state steered ONTO a bound lands on it to the accuracy of the bounded
            # solve, which must not count as outside (OSQP itself accepts 1e-3).
            xlo, xhi = db["xbox_np"]
            start = x_out[:T]
            if (start < xlo).any() or (start > xhi).any():
                raise ValueError(TVLQR_FAILED)
        self._last_descent_cost = cost
        self._last_descent = (x_out, u_out, x_out.copy(), u_out.copy())
        return x_out, u_out

    def profile_descent(self, x_trj=None, u_trj=None, repeats=5):
        """Per-phase device times of one descent from (x_trj, u_trj) (default: the current trajectory), in ms:
        the phases run one after the other on the current stream with CUDA events between them — linearization
        (one un-pipelined pass), backward Riccati pass, closed-loop rollout, plan check — next to the wall time of
        `local_descent` itself (pipelined, graph-replayed, staging copies and the synchronising read-back
        included).  Stored in `self.timings` and returned; the solver's trajectory, cost and iteration count are not
        changed (a user `sampling` closure is called for the extra linearizations, which advances ITS random stream;
        `GaussianSampling` is stateless)."""
        T, n, m = self.T, self.dim_x, self.dim_u
        x_trj = self.x_trj if x_trj is None else x_trj
        u_trj = self.u_trj if u_trj is None else u_trj
        x_all = _device.to_device(np.asarray(x_trj, dtype=np.float64)[:T + 1])
        u_nom = _device.to_device(np.asarray(u_trj, dtype=np.float64)[:T])
        x_nom = x_all[:T]
        db = self._descent_buffers()
        prm, nprm = self.system._params()
        state = {}

        def linearize():
            state["lin"] = self._tv_matrices_device(x_nom, u_nom)

        def riccati():
            At, Bt, ct, _ = state["lin"]
            self.system.lib.call("irs_tvlqr_riccati", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                      _device.ptr(self._dQ), _device.ptr(self._dQd), _device.ptr(self._dR), _device.ptr(self._dxd), 0, 1, T,
                      _device.ptr(db["K"]), _device.ptr(db["k"]), _device.ptr(db["rstatus"]), _device.stream_ptr())

        def rollout():
            self.system.lib.call("irs_rollout_closed_loop", self.system.system_id, prm, nprm, _device.ptr(db["K"]), _device.ptr(db["k"]),
                      _device.ptr(x_all), _device.ptr(self._dxd), 0, _device.ptr(self._dQ), _device.ptr(self._dR), 1, T,
                      _device.ptr(db["x_new"]), _device.ptr(db["u_new"]), _device.ptr(db["cost"]), _device.stream_ptr())

        def plan_check():
            At, Bt, ct, _ = state["lin"]
            xlo, xhi, ulo, uhi = db["box"]
            self.system.lib.call("irs_tvlqr_plan_check", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct), _device.ptr(db["K"]),
                      _device.ptr(db["k"]), _device.ptr(db["x_new"]), _device.ptr(xlo), _device.ptr(xhi), _device.ptr(ulo),
                      _device.ptr(uhi), BOUND_TOL, 1, T, 0, _device.ptr(db["violated"]), _device.ptr(db["plan_scratch"]),
                      _device.stream_ptr())

        phases = [("linearize_ms", linearize), ("riccati_ms", riccati), ("rollout_ms", rollout)]
        if db["box"] is not None:
            phases.append(("plan_check_ms", plan_check))
        for _, fn in phases:      # warm: workspaces, first launches
            fn()
        torch.cuda.synchronize()
        out = {key: 0.0 for key, _ in phases}
        for _ in range(repeats):
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(len(phases) + 1)]
            marks[0].record()
            for i, (_, fn) in enumerate(phases):
                fn()
                marks[i + 1].record()
            torch.cuda.synchronize()
            for i, (key, _) in enumerate(phases):
                out[key] += marks[i].elapsed_time(marks[i + 1]) / repeats
        out["phases_sum_ms"] = float(sum(out[key] for key, _ in phases))
        saved = (getattr(self, "_last_descent_cost", None), getattr(self, "_last_descent", None))
        self.local_descent(x_trj, u_trj)      # warm (graph capture on the third call of a shape)
        self.local_descent(x_trj, u_trj)
        self.local_descent(x_trj, u_trj)
        t0 = time.perf_counter()
        for _ in range(repeats):
            self.local_descent(x_trj, u_trj)
        out["local_descent_wall_ms"] = (time.perf_counter() - t0) / repeats * 1e3
        self._last_descent_cost, self._last_descent = saved
        self.timings = out
        return out

    def _bounded_descent(self, db):
        """irs_lqr.py:169-184 with active bounds: a box QP over the remaining horizon at every timestep
        (ADMM, csrc/tvlqr_box.cuh), first input applied to the true dynamics."""
        T, n, m = self.T, self.dim_x, self.dim_u
        At, Bt, ct = db["lin"]
        xlo, xhi, ulo, uhi = db["box_host"]
        x0 = db["in_dev"][:n].view(1, n)
        xb, ub, cost, status, iters = box_solve_device(
            self.system, True, At.view(1, T, n, n), Bt.view(1, T, n, m), ct.view(1, T, n), self._dQ, self._dQd,
            self._dR, self.Q, self.Qd, self.R, self._dxd, 0, x0, xlo, xhi, ulo, uhi, K0=db["K"], k0=db["k"])
        if int(status.item()) != 0:
            raise ValueError(TVLQR_FAILED)
        self.bounded_admm_iterations = int(iters.item())
        return _device.to_numpy(xb[0]), _device.to_numpy(ub[0]), float(cost.item())

    # -- iteration (irs_lqr.py:188-218): runs max_iterations + 1 descents ------------------------
    def iterate(self, max_iterations, verbose=True):
        while True:
            x_trj_new, u_trj_new = self.local_descent(self.x_trj, self.u_trj)
            cost_new = self.evaluate_cost(x_trj_new, u_trj_new)

            if verbose:
                print("Iteration: {:02d} ".format(self.iter) + " || " +
                      "Current Cost: {0:05f} ".format(cost_new) + " || " +
                      "Elapsed time: {0:05f} ".format(time.time() - self.start_time))

            self.x_trj_lst.append(x_trj_new)
            self.u_trj_lst.append(u_trj_new)
            self.cost_lst.append(cost_new)

            if self.iter > max_iterations:
                break

            self.cost = cost_new
            self.x_trj = x_trj_new
            self.u_trj = u_trj_new
            self.iter += 1

        return self.x_trj, self.u_trj, self.cost


def _require_jacobian(system, solver):
    if not getattr(system, "has_jacobian", True):
        raise NotImplementedError("%s needs the Jacobian of the dynamics: %r was built without one"
                                  % (solver, getattr(system, "system_name", system)))


class IrsLqrExact(IrsLqr):
    """irs_lqr/irs_lqr_exact.py:6-31 — Jacobian at the nominal point, evaluated in fp64."""

    def __init__(self, system, params):
        _require_jacobian(system, "IrsLqrExact")
        super().__init__(system, params)

    def _tv_matrices_device(self, x_nom, u_nom):
        P, n, m = x_nom.shape[0], self.dim_x, self.dim_u
        At = _device.empty((P, n, n))
        Bt = _device.empty((P, n, m))
        ct = _device.empty((P, n))
        prm, nprm = self.system._params()
        self.system.lib.call("irs_exact_linearize", self.system.system_id, prm, nprm, _device.ptr(x_nom),
                  _device.ptr(u_nom), P, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                  _device.stream_ptr())
        status = torch.zeros((P,), dtype=torch.int32, device=x_nom.device)
        return At, Bt, ct, status


RESIDENT_BLOCKS = 740      # resident grid of the quadrotor smoothing kernel on a B200 (148 SMs x 5)


def pipeline_segments(T, chunks_per_step, forced=0, min_steps=_PIPELINE_MIN_STEPS):
    """Timestep segments [(lo, hi), ...] of a pipelined descent, LATE timesteps first, or None when one
    pass is better.  Equal segments of at most one resident grid of work items (timesteps x chunks) each;
    `forced` > 0 fixes the number of segments (tests, tuning).  Measured at BASELINE.json configs[2]
    (quadrotor, T=100, N=1e5, 25 chunks per timestep, paired sampling kernel, three streams): one pass
    420 us per descent, 3 segments 408, 4: 362, 5: 364, 6: 385; back-filled unequal segments
    (29, 29, 29, 13 timesteps: short exposed tail) 395; 1024-sample chunks (98 per timestep) 390-400."""
    if forced > 0:
        k = forced
    else:
        items = T * chunks_per_step
        if items < 2 * RESIDENT_BLOCKS:
            return None       # less than two resident grids of sampling work: nothing to hide behind
        k = min(8, -(-items // RESIDENT_BLOCKS))
    while k > 1 and T // k < min_steps:
        k -= 1
    if k < 2:
        return None
    cuts = [(i * T) // k for i in range(k + 1)]
    return [(cuts[i], cuts[i + 1]) for i in reversed(range(k))]


class _SampledIrsLqr(IrsLqr):
    order = None

    def __init__(self, system, params, sampling):
        if self.order == smoothing.FIRST_ORDER:
            _require_jacobian(system, "IrsLqrFirstOrder")
        super().__init__(system, params)
        self.sampling = sampling
        self._key_cache = None

    def _replay_noise(self, x_nom, u_nom):
        """Call the user's closure once per timestep (as the reference does) and upload."""
        xh = _device.to_numpy(x_nom)
        uh = _device.to_numpy(u_nom)
        rows = []
        for t in range(xh.shape[0]):
            dx, du = self.sampling(xh[t], uh[t], self.iter)
            rows.append(np.hstack((np.asarray(dx), np.asarray(du))).astype(np.float32))
        return _device.to_device(np.stack(rows), torch.float32)

    def _tv_matrices_device(self, x_nom, u_nom):
        s = self.sampling
        if isinstance(s, GaussianSampling):
            At, Bt, ct, status, self._ws = smoothing.linearize(
                self.system, self.order, x_nom, u_nom, s.num_samples, self._ws,
                sigma=s.sigma(self.iter), seed=s.seed, it=self.iter, stream_id=s.stream_id,
                flags=s.flags())
        else:
            noise = self._replay_noise(x_nom, u_nom)
            At, Bt, ct, status, self._ws = smoothing.linearize(
                self.system, self.order, x_nom, u_nom, noise.shape[1], self._ws, noise=noise,
                flags=self._replay_flags(noise, x_nom, u_nom))
        return At, Bt, ct, status

    def _replay_flags(self, noise, x_nom, u_nom):
        """A closure may return ABSOLUTE points instead of deltas — the reference's three_cart script does
        (three_cart_zero_order.py:43 returns projection(...), SURVEY Appendix A-5), and the solver uses them
        literally.  Points that lie closer to the nominal than to the origin are accumulated relative to
        the nominal (IRS_CENTERED: the fit is the same least squares, shifted back in fp64), because an fp32
        Gram of the absolute points loses the sample spread once |xbar| >> sigma."""
        if self.order != smoothing.ZERO_ORDER or not getattr(self.system, "centered_capable", False):
            return 0
        mean = noise.to(torch.float64).mean(dim=1)
        nominal = torch.cat((x_nom, u_nom), dim=1)
        closer_to_nominal = float((mean - nominal).abs().sum().item()) < float(mean.abs().sum().item())
        return smoothing.FLAG_CENTERED if closer_to_nominal else 0

    def _pipeline_segments(self):
        """Timestep segments [(lo, hi), ...], late timesteps first, or None for the one-pass sequence.
        The backward Riccati pass needs the late timesteps first, so the horizon is linearized in a
        few launches from the back and each segment's fit and Riccati steps run on a second stream
        while the next segment is still sampling: the sequential pass hides behind the smoothing
        kernel instead of following it.  A segment is sized to about one resident grid of the
        smoothing kernel (740 blocks on a B200; a launch of fewer work items than resident blocks
        takes one item-time whatever its size, one with a few more takes two: measured on the
        quadrotor, T=100, N=1e5 with 592 resident blocks, five segments of 500 items 470 us per descent,
        three 495, four — 625 items, a second wave of 33 — 504, ten 600, one pass 515).  Results are
        bit-identical to the one-pass sequence (global point index in the Philox counter, carried
        (P, p) between segments)."""
        n, m, T = self.dim_x, self.dim_u, self.T
        if not _USE_PIPELINE or not isinstance(self.sampling, GaussianSampling) or n % 2 or m % 2 \
                or not self.system.riccati_segments:
            return None
        C, _ = smoothing.plan(self.system.system_id, self.order, T, self.sampling.num_samples, lib=self.system.lib)
        return pipeline_segments(T, C, _PIPELINE_SEGMENTS)

    def _linearize_and_riccati(self, db, x_nom, u_nom):
        segs = self._pipeline_segments()
        if segs is None:
            return super()._linearize_and_riccati(db, x_nom, u_nom)
        s = self.sampling
        T, n, m = self.T, self.dim_x, self.dim_u
        key = (self.system.system_key, self.order, T, s.num_samples)
        if self._ws is None or self._ws.key != key:
            self._ws = smoothing.Workspace(self.system, self.order, T, s.num_samples)
        ws = self._ws
        if "carry" not in db:
            db["carry"] = _device.empty((n * n + n,))
            db["side"] = torch.cuda.Stream(priority=-1)        # the sequential Riccati chain
            db["fin"] = torch.cuda.Stream(priority=-1)         # the segment fits
        main, side, fin = torch.cuda.current_stream(), db["side"], db["fin"]
        sig = s.sigma(self.iter)
        # three streams: sampling launches back to back on the main stream; each segment's fit starts as
        # soon as its samples are there (it does not wait for the previous segment's Riccati steps); the
        # Riccati segments chain on their own stream, each behind its fit.  With the paired sampling kernel
        # the backward pass (T x 1.3 us, sequential) is as long as the sampling itself, so it is the chain
        # that must never wait for anything but its inputs.
        for lo, hi in segs:
            smoothing.accumulate(self.system, self.order, x_nom, u_nom, s.num_samples, ws, sigma=sig,
                                 seed=s.seed, it=self.iter, stream_id=s.stream_id, flags=s.flags(),
                                 point_range=(lo, hi))
            sampled = torch.cuda.Event()
            sampled.record(main)
            fin.wait_event(sampled)
            with torch.cuda.stream(fin):
                smoothing.finalize(self.system, self.order, x_nom, u_nom, ws, s.num_samples, point_range=(lo, hi))
                fitted = torch.cuda.Event()
                fitted.record(fin)
            side.wait_event(fitted)
            with torch.cuda.stream(side):
                self.system.lib.call("irs_tvlqr_riccati_segment", n, m, _device.ptr(ws.At), _device.ptr(ws.Bt),
                          _device.ptr(ws.ct), _device.ptr(self._dQ), _device.ptr(self._dQd),
                          _device.ptr(self._dR), _device.ptr(self._dxd), 0, 1, T, lo, hi,
                          _device.ptr(db["carry"]), _device.ptr(db["K"]), _device.ptr(db["k"]),
                          _device.ptr(db["rstatus"]), _device.stream_ptr())
        done = torch.cuda.Event()
        done.record(side)
        main.wait_event(done)
        return ws.At, ws.Bt, ws.ct, ws.status

    def _graph_key(self):
        s = self.sampling
        if not isinstance(s, GaussianSampling):
            return None           # a Python closure is called T times per iteration: nothing to replay
        # the captured kernels bake the system parameters: a changed parameter re-captures
        prm = self.system.device_params()
        c = self._key_cache
        if c is None or c[0] != prm or c[1] != (s.num_samples, s.flags()):
            c = (prm, (s.num_samples, s.flags()),
                 (self.system.system_key, self.order, self.T, s.num_samples, s.flags(), tuple(float(v) for v in prm)))
            self._key_cache = c
        return c[2]

    def _graph_update(self, graph):
        s = self.sampling
        _, sig_ptr = s.sigma32(self.iter)
        self.system.lib.call("irs_graph_update_smoothing", graph, sig_ptr, s.seed, int(self.iter), s.stream_id)

    def _enqueue_linearize(self, ws):
        s = self.sampling
        ws.enqueue_upload()
        smoothing.accumulate(self.system, self.order, ws.x_nom, ws.u_nom, s.num_samples, ws,
                             sigma=s.sigma(self.iter), seed=s.seed, it=self.iter, stream_id=s.stream_id,
                             flags=s.flags())
        smoothing.finalize(self.system, self.order, ws.x_nom, ws.u_nom, ws, s.num_samples)
        ws.enqueue_download()

    def get_TV_matrices(self, x_trj, u_trj):
        """numpy in, numpy out: one pinned H2D copy of [x_nom | u_nom], the kernels, one D2H copy
        of [At | Bt | ct | status] — replayed from a CUDA graph once warm."""
        s = self.sampling
        if not isinstance(s, GaussianSampling):
            return super().get_TV_matrices(x_trj, u_trj)
        key = (self.system.system_key, self.order, self.T, s.num_samples)
        if self._ws is None or self._ws.key != key:
            self._ws = smoothing.Workspace(self.system, self.order, self.T, s.num_samples)
        ws = self._ws
        ws.stage_nominal(x_trj, u_trj)
        self._run("linearize", lambda: self._enqueue_linearize(ws))
        At, Bt, ct, status = ws.read_download()
        smoothing.check_status(status)
        return At, Bt, ct

    def _io_bytes(self):
        if self._ws is None:
            return super()._io_bytes()
        return self._ws.h2d_bytes(), self._ws.d2h_bytes()


class IrsLqrFirstOrder(_SampledIrsLqr):
    """irs_lqr/irs_lqr_first_order.py:6-54 — averaged Jacobians at the perturbed points."""
    order = smoothing.FIRST_ORDER


class IrsLqrZeroOrder(_SampledIrsLqr):
    """irs_lqr/irs_lqr_zero_order.py:5-63 — least-squares fit of sampled dynamics."""
    order = smoothing.ZERO_ORDER

    def compute_least_squares(self, dxdu, deltaf):
        """irs_lqr_zero_order.py:27-36: (Ahat, Bhat) = lstsq(dxdu, deltaf)^T split, on explicit samples.
        The library's own kernels: the packed fp64 Gram block (irs_gram_block_f64) and the Cholesky fit of
        the finalize kernel (normal equations: identical to lstsq for full column rank; a rank-deficient
        sample set raises LinAlgError instead of returning the min-norm solution)."""
        dxdu = np.ascontiguousarray(np.asarray(dxdu, dtype=np.float64))
        deltaf = np.ascontiguousarray(np.asarray(deltaf, dtype=np.float64))
        n, m = self.dim_x, self.dim_u
        d = n + m
        if dxdu.ndim != 2 or dxdu.shape[1] != d or deltaf.shape != (dxdu.shape[0], n):
            raise ValueError("expected dxdu [N, %d] and deltaf [N, %d]" % (d, n))
        N = dxdu.shape[0]
        Z, F = _device.to_device(dxdu), _device.to_device(deltaf)
        width = self.system.lib.handle().irs_partial_width(self.system.system_id, smoothing.ZERO_ORDER)
        block = torch.zeros((1, width), dtype=torch.float64, device=Z.device)
        self.system.lib.call("irs_gram_block_f64", n, m, _device.ptr(Z), _device.ptr(F), N, _device.ptr(block),
                  _device.stream_ptr())
        zero_x, zero_u = torch.zeros((1, n), dtype=torch.float64, device=Z.device), \
            torch.zeros((1, m), dtype=torch.float64, device=Z.device)
        At, Bt, ct = _device.empty((1, n, n)), _device.empty((1, n, m)), _device.empty((1, n))
        status = _device.empty((1,), torch.int32)
        prm, nprm = self.system._params()
        self.system.lib.call("irs_smooth_finalize", self.system.system_id, prm, nprm, smoothing.ZERO_ORDER, _device.ptr(zero_x),
                  _device.ptr(zero_u), 1, 1, None, _device.ptr(block), 1, 0, float(N), 0, _device.ptr(At),
                  _device.ptr(Bt), _device.ptr(ct), _device.ptr(status), _device.stream_ptr())
        smoothing.check_status(status)
        return _device.to_numpy(At[0]), _device.to_numpy(Bt[0])
