"""Cross-entropy-method baseline with the reference's call surface (irs_lqr/cem.py:7-216).

`CemParameters` / `CrossEntropyMethod` keep the reference's names, attributes and iteration
bookkeeping.  The data-parallel part of `local_descent` (cem.py:151-184) — rolling out and
costing `batch_size` candidate input trajectories — is ONE launch of the batched open-loop
rollout kernel (irs_rollout_open_loop, one warp per candidate, fp64) instead of a Python loop
over candidates and timesteps; the elite selection (`np.argpartition`, :175) and the mean / std
refit (:180-182) run on the device too (csrc/cem.cuh: rank + refit kernels), followed by the rollout of
the new mean, so one CEM step uploads the candidates once and reads back T*(n+2m) numbers.  Candidate
sampling stays `np.random.normal` on the host, exactly as in the reference (cem.py:162-163: same
global numpy RNG stream, so a seeded run draws the same candidates).
"""
import time

import numpy as np
import torch

from . import _device, _lib
from .dynamical_system import CudaDynamicalSystem


class CemParameters:
    """Attribute bag, irs_lqr/cem.py:7-33."""

    def __init__(self):
        self.Q = None
        self.Qd = None
        self.R = None
        self.x0 = None
        self.xd_trj = None
        self.u_trj_initial = None
        self.n_elite = None
        self.batch_size = None
        self.elite_frac = None
        self.initial_std = None   # dim u array of initial stds.


class CrossEntropyMethod:
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
        self.n_elite = params.n_elite
        self.batch_size = params.batch_size
        self.elite_frac = params.elite_frac
        self.initial_std = params.initial_std

        self.T = self.u_trj.shape[0]
        self.dim_x = self.system.dim_x
        self.dim_u = self.system.dim_u
        self._dQ = _device.to_device(np.asarray(self.Q, dtype=np.float64))
        self._dR = _device.to_device(np.asarray(self.R, dtype=np.float64))
        self._dxd = _device.to_device(np.asarray(self.xd_trj, dtype=np.float64)[:self.T + 1])

        self.x_trj = self.rollout(self.x0, self.u_trj)
        self.cost = self.evaluate_cost(self.x_trj, self.u_trj)
        self.std_trj = np.tile(self.initial_std, (self.T, 1))

        self.x_trj_lst = [self.x_trj]
        self.u_trj_lst = [self.u_trj]
        self.cost_lst = [self.cost]
        self.start_time = time.time()
        self.iter = 1

    # -- validation (cem.py:76-107, same messages) ---------------------------------------------
    def check_valid_system(self, system):
        if system.dim_x == 0:
            raise RuntimeError("System has zero states. Did you forget to set dim_x?")
        elif system.dim_u == 0:
            raise RuntimeError("System has zero inputs. Did you forget to set dim_u?")
        if not isinstance(system, CudaDynamicalSystem):
            raise RuntimeError("Could not evaluate dynamics. irs_mpc_b200 runs the dynamics as CUDA "
                               "functors: the system must derive from CudaDynamicalSystem.")
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

    # -- batched rollout + cost (cem.py:109-149 for every candidate at once) --------------------
    def rollout_batch(self, x0, u_candidates):
        """u_candidates [B,T,m] -> (x_trj [B,T+1,n], cost [B]) numpy float64."""
        u = np.ascontiguousarray(np.asarray(u_candidates, dtype=np.float64))
        B = u.shape[0]
        ud = _device.to_device(u)
        x0d = _device.to_device(np.tile(np.asarray(x0, dtype=np.float64), (B, 1)))
        x_trj = _device.empty((B, self.T + 1, self.dim_x))
        cost = _device.empty((B,))
        prm, nprm = self.system._params()
        self.system.lib.call("irs_rollout_open_loop", self.system.system_id, prm, nprm, _device.ptr(ud),
                  _device.ptr(x0d), _device.ptr(self._dxd), 0, _device.ptr(self._dQ),
                  _device.ptr(self._dR), B, self.T, _device.ptr(x_trj), _device.ptr(cost),
                  _device.stream_ptr())
        return _device.to_numpy(x_trj), _device.to_numpy(cost)

    def rollout(self, x0, u_trj):
        return self.rollout_batch(x0, np.asarray(u_trj, dtype=np.float64)[None])[0][0]

    def evaluate_cost(self, x_trj, u_trj):
        import torch
        x = _device.to_device(np.asarray(x_trj, dtype=np.float64).reshape(1, self.T + 1, self.dim_x))
        u = _device.to_device(np.asarray(u_trj, dtype=np.float64).reshape(1, self.T, self.dim_u))
        cost = _device.empty((1,))
        self.system.lib.call("irs_evaluate_cost", self.dim_x, self.dim_u, _device.ptr(x), _device.ptr(u),
                  _device.ptr(self._dxd), 0, _device.ptr(self._dQ), _device.ptr(self._dR), 1, self.T,
                  _device.ptr(cost), _device.stream_ptr())
        return float(cost.item())

    def get_TV_matrices(self, x_trj, u_trj):
        raise NotImplementedError("This class is virtual.")

    # -- one CEM step (cem.py:151-184) --------------------------------------------------------------
    def local_descent(self, x_trj, u_trj):
        B, T, n, m = self.batch_size, self.T, self.dim_x, self.dim_u
        # 1. candidates around the current mean (same numpy call as the reference: same stream)
        u_trj_candidates = np.random.normal(u_trj, self.std_trj, (B, T, m))
        ud = _device.to_device(np.ascontiguousarray(u_trj_candidates, dtype=np.float64))
        x0d = _device.to_device(np.tile(np.asarray(self.x0, dtype=np.float64), (B, 1)))
        x_cand = _device.empty((B, T + 1, n))
        cost = _device.empty((B,))
        prm, nprm = self.system._params()
        # 2. roll all of them out and cost them: one kernel launch
        self.system.lib.call("irs_rollout_open_loop", self.system.system_id, prm, nprm, _device.ptr(ud),
                  _device.ptr(x0d), _device.ptr(self._dxd), 0, _device.ptr(self._dQ),
                  _device.ptr(self._dR), B, T, _device.ptr(x_cand), _device.ptr(cost), _device.stream_ptr())
        # 3.-4. the n_elite cheapest, mean and std over them — on the device; out = [mean | std | x of the mean]
        elite = _device.empty((B,), torch.int32)
        out = _device.empty((2 * T * m + (T + 1) * n + 1,))
        mean, std = out[:T * m].view(1, T, m), out[T * m:2 * T * m]
        x_new = out[2 * T * m:2 * T * m + (T + 1) * n].view(1, T + 1, n)
        self.system.lib.call("irs_cem_refit", _device.ptr(cost), _device.ptr(ud), B, T, m, int(self.n_elite),
                  _device.ptr(elite), _device.ptr(mean), _device.ptr(std), _device.stream_ptr())
        # rollout of the new mean (cem.py:183)
        self.system.lib.call("irs_rollout_open_loop", self.system.system_id, prm, nprm, _device.ptr(mean),
                  _device.ptr(x0d), _device.ptr(self._dxd), 0, _device.ptr(self._dQ),
                  _device.ptr(self._dR), 1, T, _device.ptr(x_new), _device.ptr(out[-1:]), _device.stream_ptr())
        h = _device.to_numpy(out)
        self.std_trj = h[T * m:2 * T * m].reshape(T, m).copy()
        self.last_elite = elite                      # device mask of the step (diagnostics / tests)
        return h[2 * T * m:2 * T * m + (T + 1) * n].reshape(T + 1, n).copy(), h[:T * m].reshape(T, m).copy()

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
