"""Batched iRS-LQR: I independent MPC instances of the same system stepped together.

BASELINE.json configs[4] ("4096 independent quadrotor MPC instances, batched TVLQR Riccati +
smoothing, instances sharded over 8 B200").  The reference has no such class — it runs one
`IrsLqr` object per problem (irs_lqr/irs_lqr.py:34-71); this is the same algorithm
(`local_descent`, irs_lqr.py:148-186, and `iterate`, :188-218) with a leading instance axis:

  * smoothing: the I*T nominal points are one launch of the fused kernels (point index
    b*T + t in the Philox counter, so instance b alone with p0 = b*T draws the same noise);
  * TVLQR: one warp per instance runs the affine Riccati recursion, one warp per instance the
    closed-loop rollout on the true dynamics — the sequential pass is never split;
  * everything stays on the device between iterations; only the I costs travel to the host.

Instances shard trivially over GPUs: each rank constructs the object with its slice of
(x0, xd_trj, u_trj_initial) and `instance_offset` = index of its first instance; no collective is
needed on the data path (bench.py gathers the costs at the end).
"""
import numpy as np
import torch

from . import _device, _lib, smoothing
from .dynamical_system import CudaDynamicalSystem
from .sampling import GaussianSampling
from .tv_lqr import TVLQR_FAILED


class BatchedIrsLqrZeroOrder:
    order = smoothing.ZERO_ORDER

    def __init__(self, system, Q, Qd, R, x0, xd_trj, u_trj_initial, sampling, instance_offset=0,
                 xbound=None, ubound=None):
        """x0 [I,n]; xd_trj [I,T+1,n] or [T+1,n] (shared); u_trj_initial [I,T,m] or [T,m].
        xbound [2,n] / ubound [2,m]: the reference's IrsLqrParameters.xbound / ubound (irs_lqr.py:160-167), the
        same box for every instance.  The batched path runs the one-pass Riccati descent, which is the
        reference's result while no planned trajectory touches a bound; with bounds given, every descent is
        followed by the plan check of all instances x start times (irs_tvlqr_plan_check) and `check()` raises
        the reference's ValueError for instances whose QPs would have had an active bound (e.g. a quadrotor
        plan through the +-pi/2 pitch bound that guards the 1/cos(pitch) singularity) — run those through
        IrsLqrZeroOrder, which solves the bounded QPs."""
        if not isinstance(system, CudaDynamicalSystem):
            raise RuntimeError("the system must derive from CudaDynamicalSystem (no CPU fallback)")
        if not isinstance(sampling, GaussianSampling):
            raise RuntimeError("batched instances use the in-kernel Philox sampler (GaussianSampling)")
        self.system, self.sampling = system, sampling
        n, m = system.dim_x, system.dim_u
        x0 = np.asarray(x0, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != n:
            raise RuntimeError("x0 must be [I, dim_x]")
        self.I = x0.shape[0]
        u0 = np.asarray(u_trj_initial, dtype=np.float64)
        if u0.ndim == 2:
            u0 = np.broadcast_to(u0, (self.I,) + u0.shape)
        self.T = u0.shape[1]
        xd = np.asarray(xd_trj, dtype=np.float64)
        self.xd_shared = xd.ndim == 2
        if np.asarray(Q).shape != (n, n) or np.asarray(Qd).shape != (n, n) or np.asarray(R).shape != (m, m):
            raise RuntimeError("Q, Qd must be dim_x x dim_x and R dim_u x dim_u")
        self.dim_x, self.dim_u = n, m
        self.instance_offset = int(instance_offset)
        self._dQ, self._dQd, self._dR = _device.to_device(Q), _device.to_device(Qd), _device.to_device(R)
        self._dxd = _device.to_device(np.ascontiguousarray(xd[..., :self.T + 1, :]))
        self._xd_stride = 0 if self.xd_shared else (self.T + 1) * n
        I, T = self.I, self.T
        self._x0 = _device.to_device(x0)
        self.u_trj = _device.to_device(np.ascontiguousarray(u0))
        self.x_trj = _device.empty((I, T + 1, n))
        self.cost = _device.empty((I,))
        self._x_new = _device.empty((I, T + 1, n))
        self._u_new = _device.empty((I, T, m))
        self._cost_new = _device.empty((I,))
        self._K = _device.empty((I, T, m, n))
        self._k = _device.empty((I, T, m))
        self._rstatus = _device.empty((I,), torch.int32)
        self._ws = smoothing.Workspace(system, self.order, I * T, sampling.num_samples)
        self._box = None
        if xbound is not None or ubound is not None:
            if I > 65535:
                raise RuntimeError("the plan check supports at most 65535 instances per object")
            big = 1e30
            xlo, xhi = ((np.asarray(xbound[0], dtype=np.float64), np.asarray(xbound[1], dtype=np.float64))
                        if xbound is not None else (-big * np.ones(n), big * np.ones(n)))
            ulo, uhi = ((np.asarray(ubound[0], dtype=np.float64), np.asarray(ubound[1], dtype=np.float64))
                        if ubound is not None else (-big * np.ones(m), big * np.ones(m)))
            self._box = tuple(_device.to_device(np.ascontiguousarray(v)) for v in (xlo, xhi, ulo, uhi))
            self._plan_scratch = _device.empty((I * T * (n + m) * (n + 1),))
            self._violated = _device.empty((I,), torch.int32)
        self._rollout_open(self._x0, self.u_trj, self.x_trj, self.cost)
        self.iter = 1
        self.cost_lst = [_device.to_numpy(self.cost)]

    # -- device launches ------------------------------------------------------------------------
    def _rollout_open(self, x0, u, x_out, cost_out):
        prm, nprm = self.system._params()
        self.system.lib.call("irs_rollout_open_loop", self.system.system_id, prm, nprm, _device.ptr(u),
                  _device.ptr(x0), _device.ptr(self._dxd), self._xd_stride, _device.ptr(self._dQ),
                  _device.ptr(self._dR), self.I, self.T, _device.ptr(x_out), _device.ptr(cost_out),
                  _device.stream_ptr())

    def linearize(self):
        """(At [I,T,n,n], Bt [I,T,n,m], ct [I,T,n], status [I*T]) on the device for the current
        nominal trajectories (IrsLqrZeroOrder.get_TV_matrices for every instance at once)."""
        I, T, n, m = self.I, self.T, self.dim_x, self.dim_u
        s = self.sampling
        x_nom = self.x_trj[:, :T, :].contiguous().view(I * T, n)
        u_nom = self.u_trj.view(I * T, m)
        smoothing.accumulate(self.system, self.order, x_nom, u_nom, s.num_samples, self._ws,
                             sigma=s.sigma(self.iter), seed=s.seed, it=self.iter, stream_id=s.stream_id,
                             p0=self.instance_offset * T, flags=s.flags())
        At, Bt, ct, status = smoothing.finalize(self.system, self.order, x_nom, u_nom, self._ws,
                                                s.num_samples)
        return At.view(I, T, n, n), Bt.view(I, T, n, m), ct.view(I, T, n), status

    def local_descent(self):
        """One descent of every instance from its current trajectory; returns device tensors
        (x_new [I,T+1,n], u_new [I,T,m], cost_new [I]).  No host synchronisation."""
        I, T, n, m = self.I, self.T, self.dim_x, self.dim_u
        At, Bt, ct, self._sstatus = self.linearize()
        self.system.lib.call("irs_tvlqr_riccati", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                  _device.ptr(self._dQ), _device.ptr(self._dQd), _device.ptr(self._dR),
                  _device.ptr(self._dxd), self._xd_stride, I, T, _device.ptr(self._K),
                  _device.ptr(self._k), _device.ptr(self._rstatus), _device.stream_ptr())
        prm, nprm = self.system._params()
        self.system.lib.call("irs_rollout_closed_loop", self.system.system_id, prm, nprm, _device.ptr(self._K),
                  _device.ptr(self._k), _device.ptr(self.x_trj[:, 0, :].contiguous()),
                  _device.ptr(self._dxd), self._xd_stride, _device.ptr(self._dQ), _device.ptr(self._dR),
                  I, T, _device.ptr(self._x_new), _device.ptr(self._u_new), _device.ptr(self._cost_new),
                  _device.stream_ptr())
        if self._box is not None:
            from .tv_lqr import BOUND_TOL
            xlo, xhi, ulo, uhi = self._box
            self.system.lib.call("irs_tvlqr_plan_check", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                      _device.ptr(self._K), _device.ptr(self._k), _device.ptr(self._x_new), _device.ptr(xlo),
                      _device.ptr(xhi), _device.ptr(ulo), _device.ptr(uhi), BOUND_TOL, I, T, 0,
                      _device.ptr(self._violated), _device.ptr(self._plan_scratch), _device.stream_ptr())
        return self._x_new, self._u_new, self._cost_new

    def check(self):
        """Synchronising status check (rank-deficient fits, failed Riccati passes)."""
        smoothing.check_status(self._sstatus)
        bad = int(self._rstatus.sum().item())
        if bad or not bool(torch.isfinite(self._cost_new).all().item()):
            raise ValueError(TVLQR_FAILED)
        if self._box is not None and int(self._violated.sum().item()):
            hit = torch.nonzero(self._violated).flatten().tolist()
            raise ValueError(TVLQR_FAILED + " A planned trajectory of %d instance(s) touches xbound / ubound "
                             "(first: %s, offsets into this object): the batched path does not solve bounded QPs; "
                             "run these instances through IrsLqrZeroOrder." % (len(hit), hit[:8]))

    def iterate(self, max_iterations, verbose=False):
        """irs_lqr.py:188-218 for every instance: max_iterations + 1 descents, the state keeps the
        max_iterations-th.  Returns (x_trj, u_trj, cost) as numpy arrays."""
        while True:
            x_new, u_new, cost_new = self.local_descent()
            self.check()
            c = _device.to_numpy(cost_new)
            if verbose:
                print("Iteration: {:02d}  || mean cost over {} instances: {:05f}".format(
                    self.iter, self.I, float(c.mean())))
            self.cost_lst.append(c)
            if self.iter > max_iterations:
                break
            self.x_trj, self._x_new = x_new, self.x_trj
            self.u_trj, self._u_new = u_new, self.u_trj
            self.cost, self._cost_new = cost_new, self.cost
            self.iter += 1
        return _device.to_numpy(self.x_trj), _device.to_numpy(self.u_trj), _device.to_numpy(self.cost)
