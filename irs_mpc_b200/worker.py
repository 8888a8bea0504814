"""Worker wire protocol of the reference's task farm, answered from a GPU (SURVEY.md section 8(f)-4).

The reference distributes the linearization of a trajectory over worker PROCESSES: the solver binds a PUSH
socket on tcp://*:5557 and a PULL socket on tcp://*:5558 (irs_lqr/irs_lqr_quasistatic.py:118-126), sends one task
per stride of timesteps — a two-frame message, JSON metadata {dtype, shape, t, n_samples, std} followed by the raw
array of nominal points [k, n_x + n_u] (zmq_parallel_cmp/array_io.py:6-18, irs_lqr_quasistatic.py:240-258) — and
collects [k, n_x, n_x + n_u] blocks [A | B] tagged with the same `t` list (:259-263).  A worker connects PULL to
5557 and PUSH to 5558, and for every task calls `calc_AB_batch(x_nominals, u_nominals, n_samples, std_u, mode)`
(examples/planar_hand/planar_hand_worker.py:19-80; quasistatic_dynamics.py:210-240), replying with
`send_array(sender, A=ABhat, t=t_list, n_samples=-1, std=[-1])`.

`GpuLinearizationWorker` is such a worker for any `CudaDynamicalSystem`: one process, one GPU, the k nominal points
of a task are ONE launch of the smoothing kernels.  Modes as in quasistatic_dynamics.py:217-236:
  "zero_order_AB"  least-squares fit of [A | B] on N samples (calc_AB_zero_order, :268-300; the reference's
                   ridge rows, damp = 1e-2, are not added: the in-kernel fit is the plain lstsq of
                   irs_lqr_zero_order.py:27-36)
  "first_order"    mean of the Jacobians at the samples (calc_AB_first_order, :193-208)
  "exact"          Jacobian at the nominal point (calc_AB_exact, :190-191)
`std` in a task is the input standard deviation (`std_u`, a scalar or n_u values); the state standard deviation is
the worker's `std_x` (the reference's calc_AB_zero_order default is 1e-3, :270); a list of n_x + n_u values is
taken as the full sigma.  The Philox counters carry the GLOBAL timestep index t, so the answer for a timestep does
not depend on how the solver strides its tasks over workers.

`send_array` / `recv_array` are the reference's framing (array_io.py:6-26), byte compatible.
"""
import numpy as np
import torch

from . import _device, smoothing
from .dynamical_system import CudaDynamicalSystem

MODES = {"zero_order_AB": smoothing.ZERO_ORDER, "first_order": smoothing.FIRST_ORDER, "exact": None}


def send_array(socket, A, t, n_samples, std, flags=0, copy=True, track=False):
    """zmq_parallel_cmp/array_io.py:6-18: JSON metadata frame, then the array bytes."""
    import zmq
    A = np.ascontiguousarray(A)
    md = dict(dtype=str(A.dtype), shape=A.shape, t=t, n_samples=n_samples, std=std)
    socket.send_json(md, flags | zmq.SNDMORE)
    return socket.send(A, flags, copy=copy, track=track)


def recv_array(socket, flags=0, copy=True, track=False):
    """zmq_parallel_cmp/array_io.py:21-26 -> (array, t, n_samples, std)."""
    md = socket.recv_json(flags=flags)
    msg = socket.recv(flags=flags, copy=copy, track=track)
    xu = np.frombuffer(memoryview(msg), dtype=md["dtype"])
    return xu.reshape(md["shape"]), md["t"], md["n_samples"], md["std"]


def contiguous_runs(t_list):
    """[(first index into t_list, length)] of the maximal runs t, t+1, t+2, ... (host logic)."""
    runs, start = [], 0
    for i in range(1, len(t_list) + 1):
        if i == len(t_list) or t_list[i] != t_list[i - 1] + 1:
            runs.append((start, i - start))
            start = i
    return runs


class GpuLinearizationWorker:
    def __init__(self, system, mode="zero_order_AB", std_x=1e-3, seed=0, iteration=1, antithetic=True,
                 pull_addr="tcp://localhost:5557", push_addr="tcp://localhost:5558", context=None):
        if not isinstance(system, CudaDynamicalSystem):
            raise RuntimeError("the system must derive from CudaDynamicalSystem (no CPU fallback)")
        if mode not in MODES:
            raise RuntimeError("AB mode %s is not supported." % mode)        # quasistatic_dynamics.py:238
        self.system, self.mode, self.order = system, mode, MODES[mode]
        n = system.dim_x
        self.std_x = np.broadcast_to(np.asarray(std_x, dtype=np.float64), (n,)).copy()
        self.seed, self.iteration = int(seed), int(iteration)
        self.flags = smoothing.FLAG_ANTITHETIC if antithetic else 0
        self.pull_addr, self.push_addr = pull_addr, push_addr
        self._context, self._ws = context, None
        self.tasks_done = 0

    # -- the computation of one task ---------------------------------------------------------------
    def sigma(self, std):
        n, m = self.system.dim_x, self.system.dim_u
        std = np.atleast_1d(np.asarray(std, dtype=np.float64))
        if std.size == n + m:
            return std.copy()
        if std.size not in (1, m):
            raise ValueError("std must hold 1, n_u = %d or n_x + n_u = %d values, got %d" % (m, n + m, std.size))
        return np.concatenate((self.std_x, np.broadcast_to(std, (m,))))

    def calc_AB_batch(self, x_nominals, u_nominals, n_samples, std, t_list=None):
        """quasistatic_dynamics.py:210-240 on the GPU: [k, n_x, n_x + n_u] float64.  t_list: the trajectory
        indices of the points (Philox point index); default 0 .. k-1."""
        s = self.system
        n, m = s.dim_x, s.dim_u
        x = np.ascontiguousarray(np.asarray(x_nominals, dtype=np.float64))
        u = np.ascontiguousarray(np.asarray(u_nominals, dtype=np.float64))
        if x.ndim != 2 or u.ndim != 2 or x.shape[1] != n or u.shape[1] != m or x.shape[0] != u.shape[0]:
            raise ValueError("expected nominal points [k, %d] and [k, %d], got %s and %s" % (n, m, x.shape, u.shape))
        k = x.shape[0]
        t_list = list(range(k)) if t_list is None else [int(t) for t in t_list]
        if len(t_list) != k:
            raise ValueError("t must name every nominal point (%d points, %d indices)" % (k, len(t_list)))
        out = np.zeros((k, n, n + m))
        if k == 0:
            return out
        xd, ud = _device.to_device(x), _device.to_device(u)
        if self.order is None:
            At, Bt, ct = _device.empty((k, n, n)), _device.empty((k, n, m)), _device.empty((k, n))
            prm, nprm = s._params()
            s.lib.call("irs_exact_linearize", s.system_id, prm, nprm, _device.ptr(xd), _device.ptr(ud), k,
                      _device.ptr(At), _device.ptr(Bt), _device.ptr(ct), _device.stream_ptr())
            out[:, :, :n], out[:, :, n:] = _device.to_numpy(At), _device.to_numpy(Bt)
            return out
        N = int(n_samples)
        if N < 1:
            raise ValueError("n_samples must be positive")
        sigma = self.sigma(std)
        for first, length in contiguous_runs(t_list):
            if self._ws is None or self._ws.key != (s.system_id, self.order, length, N):
                self._ws = smoothing.Workspace(s, self.order, length, N)
            ws = self._ws
            xs, us = xd[first:first + length], ud[first:first + length]
            smoothing.accumulate(s, self.order, xs, us, N, ws, sigma=sigma, seed=self.seed, it=self.iteration,
                                 p0=t_list[first], flags=self.flags)
            At, Bt, _, status = smoothing.finalize(s, self.order, xs, us, ws, N)
            smoothing.check_status(status)
            out[first:first + length, :, :n] = _device.to_numpy(At)
            out[first:first + length, :, n:] = _device.to_numpy(Bt)
        return out

    # -- the wire loop (planar_hand_worker.py:19-80) ---------------------------------------------------
    def serve(self, max_tasks=None, poll_ms=None):
        """Process tasks until max_tasks are done (None: forever).  poll_ms: return when no task arrives for that
        long (tests).  Returns the number of tasks processed by this call."""
        import zmq
        context = self._context if self._context is not None else zmq.Context.instance()
        receiver = context.socket(zmq.PULL)
        receiver.connect(self.pull_addr)
        sender = context.socket(zmq.PUSH)
        sender.connect(self.push_addr)
        done = 0
        try:
            while max_tasks is None or done < max_tasks:
                if poll_ms is not None and not receiver.poll(poll_ms):
                    break
                x_u_nominal, t_list, n_samples, std = recv_array(receiver)
                assert len(x_u_nominal.shape) == 2
                n = self.system.dim_x
                ABhat = self.calc_AB_batch(x_u_nominal[:, :n], x_u_nominal[:, n:], n_samples, std, t_list)
                send_array(sender, A=ABhat, t=t_list, n_samples=-1, std=[-1])
                done += 1
                self.tasks_done += 1
        finally:
            receiver.close(linger=0)
            sender.close(linger=1000)
        return done


def linearize_with_workers(sender, receiver, x_trj, u_trj, n_samples, std, stride):
    """The solver side, irs_lqr_quasistatic.py:228-263: one task per `stride` timesteps over bound PUSH / PULL
    sockets, blocks written back by their `t` lists.  Returns (At [T,n,n], Bt [T,n,m])."""
    x_trj, u_trj = np.asarray(x_trj, dtype=np.float64), np.asarray(u_trj, dtype=np.float64)
    T, n, m = u_trj.shape[0], x_trj.shape[1], u_trj.shape[1]
    At, Bt = np.zeros((T, n, n)), np.zeros((T, n, m))
    sent = 0
    for t in range(0, T, stride):
        t1 = min(t + stride, T)
        x_u = np.zeros((t1 - t, n + m))
        x_u[:, :n] = x_trj[t:t1]
        x_u[:, n:] = u_trj[t:t1]
        send_array(sender, x_u, t=np.arange(t, t1).tolist(), n_samples=n_samples, std=np.asarray(std).tolist())
        sent += 1
    for _ in range(sent):
        ABhat, t_list, _, _ = recv_array(receiver)
        At[t_list] = ABhat[:, :, :n]
        Bt[t_list] = ABhat[:, :, n:]
    return At, Bt
