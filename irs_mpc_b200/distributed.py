"""Multi-GPU smoothing: one process per GPU (torchrun), torch.distributed for the plumbing.

The reference's only "distributed backend" is a ZeroMQ PUSH/PULL task farm over timesteps
(irs_lqr/irs_lqr_quasistatic.py:228-273, zmq_parallel_cmp/array_io.py:6-26).  Here:

* timestep sharding (`linearize_t`): rank r owns the nominal points [r*ceil(T/W), ...); every
  rank runs the fused kernels on its slice with the GLOBAL point index in the Philox counter and
  the per-point blocks [A_t | B_t | c_t] are all-gathered (n*(n+m+1) doubles per step).  Results
  are bit-identical to the single-GPU run because the per-point reduction order is unchanged.
* sample sharding (`linearize_n`): every rank owns all T points and a slice of the samples
  (global sample index in the Philox counter); the chunk-reduced fp64 Gram blocks [T, width] are
  all-gathered and every rank sums them in rank order and solves — deterministic, identical on
  all ranks, and the exchange is T*width doubles per rank.
The sequential Riccati pass is never split (replicated on every rank).

The gather helpers are backend agnostic (NCCL on GPUs, gloo in the CPU tests).
"""
import numpy as np
import torch
import torch.distributed as dist

from . import _device, _lib, smoothing
from ._graph import GraphRunner


def shard_range(total, world, rank):
    """Contiguous ceil-split: [start, stop) of `total` items owned by `rank` (may be empty)."""
    per = (total + world - 1) // world
    start = min(rank * per, total)
    stop = min(start + per, total)
    return start, stop, per


def pack_abc(At, Bt, ct):
    """[L,n,n], [L,n,m], [L,n] -> [L, n*(n+m+1)] (row-major [A|B|c] per step)."""
    L, n = ct.shape
    m = Bt.shape[2]
    return torch.cat((At.reshape(L, n * n), Bt.reshape(L, n * m), ct.reshape(L, n)), dim=1)


def unpack_abc(packed, n, m):
    L = packed.shape[0]
    At = packed[:, :n * n].reshape(L, n, n)
    Bt = packed[:, n * n:n * n + n * m].reshape(L, n, m)
    ct = packed[:, n * n + n * m:].reshape(L, n)
    return At, Bt, ct


def gather_rows(local, total, group=None):
    """All-gather row blocks of a ceil-split [total, w] array.  `local` holds this rank's rows
    (possibly fewer than ceil(total/W), possibly zero); returns the full [total, w] tensor."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    start, stop, per = shard_range(total, world, rank)
    assert local.shape[0] == stop - start, (local.shape, start, stop)
    w = local.shape[1]
    padded = torch.zeros((per, w), dtype=local.dtype, device=local.device)
    if stop > start:
        padded[:stop - start].copy_(local)
    out = torch.empty((world * per, w), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded, group=group)
    return out[:total]


def gather_ranks(local, group=None):
    """All-gather equally shaped blocks: [*shape] -> [W, *shape]."""
    world = dist.get_world_size(group)
    flat = local.contiguous().view(-1)
    out = torch.empty((world * flat.numel(),), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, flat, group=group)
    return out.view((world,) + tuple(local.shape))


class PeerExchange:
    """Exchange buffers in peer-mapped (symmetric) memory for the sample-sharded path.  The finalize
    kernel itself reduces this rank's partials of a nominal point, stores the fp64 block into every
    peer over NVLink, raises a per-point arrival flag and waits for the peers' flags of that point
    (csrc/smooth.cuh: peer_exchange_point) — reduction, all-gather and fit are ONE launch and there is
    no NCCL call on the data path.  torch's symmetric-memory allocator is used for the address
    exchange only (plumbing).

    The epoch lives in device memory and is advanced by the kernel, flags are indexed by point: a
    changed horizon (fewer or more points per call) keeps the ranks in step, and the call sequence can
    be replayed from a CUDA graph.  A peer that does not deliver within `timeout_s` makes the points
    concerned return status 2, which `smoothing.check_status` turns into a RuntimeError."""

    TIMEOUT_S = 10.0

    def __init__(self, points, width, group=None, timeout_s=None):
        import torch.distributed._symmetric_memory as symm_mem
        group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.points, self.width = int(points), int(width)
        self.slot_stride = (self.points * self.width + 15) // 16 * 16
        self.flag_stride = (self.points + 31) // 32 * 32
        self.timeout_s = float(self.TIMEOUT_S if timeout_s is None else timeout_s)
        dev = torch.device("cuda", torch.cuda.current_device())
        self.buf = symm_mem.empty((2 * self.world * self.slot_stride,), dtype=torch.float64, device=dev)
        self.flags = symm_mem.empty((self.world * self.flag_stride,), dtype=torch.int32, device=dev)
        self.buf.zero_()
        self.flags.zero_()
        self._hbuf = symm_mem.rendezvous(self.buf, group)
        self._hflags = symm_mem.rendezvous(self.flags, group)
        self.epoch = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.counter = torch.zeros((1,), dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        self._hflags.barrier()          # every rank's flags are zero before anyone raises one

    def fits(self, P, width):
        return P * width <= self.slot_stride and P <= self.flag_stride and width == self.width

    def finalize(self, system, order, x_nom, u_nom, ws, n_total):
        """Enqueue the fused reduce + exchange + fit of this step (all ranks, same order)."""
        P = x_nom.shape[0]
        prm, nprm = system._params()
        _lib.call("irs_smooth_finalize_peer", system.system_id, prm, nprm, order, _device.ptr(x_nom),
                  _device.ptr(u_nom), P, ws.C, _device.ptr(ws.partials), self._hbuf.buffer_ptrs_dev,
                  self._hflags.buffer_ptrs_dev, _device.ptr(self.epoch), _device.ptr(self.counter),
                  self.slot_stride, self.flag_stride, self.rank, self.world, self.timeout_s, float(n_total),
                  1 if ws.centered else 0, _device.ptr(ws.At), _device.ptr(ws.Bt),
                  _device.ptr(ws.ct), _device.ptr(ws.status), _device.stream_ptr())
        return ws.At, ws.Bt, ws.ct, ws.status


class TimestepGather:
    """Output buffers in peer-mapped (symmetric) memory for the timestep-sharded path: the finalize kernel
    of every rank writes the [A_t | B_t | c_t | status] blocks of ITS timesteps straight into every rank's
    buffer and the last block of each launch waits for all T arrival flags (csrc/smooth.cuh:
    write_abc_gather) — the all-gather is part of the fit kernel, two launches per step, no NCCL."""

    TIMEOUT_S = 10.0

    def __init__(self, system, T, group=None, timeout_s=None):
        import torch.distributed._symmetric_memory as symm_mem
        group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        n, m = system.dim_x, system.dim_u
        self.T, self.n, self.m = int(T), n, m
        self.out_stride = (self.T * (n * (n + m + 1) + 1) + 15) // 16 * 16
        self.timeout_s = float(self.TIMEOUT_S if timeout_s is None else timeout_s)
        dev = torch.device("cuda", torch.cuda.current_device())
        self.out = symm_mem.empty((2 * self.out_stride,), dtype=torch.float64, device=dev)
        self.flags = symm_mem.empty(((self.T + 31) // 32 * 32,), dtype=torch.int32, device=dev)
        self.out.zero_()
        self.flags.zero_()
        self._hout = symm_mem.rendezvous(self.out, group)
        self._hflags = symm_mem.rendezvous(self.flags, group)
        self.epoch = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.counter = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.calls = 0                  # host mirror of the device epoch: which parity holds the last step
        torch.cuda.synchronize()
        self._hflags.barrier()

    def enqueue(self, system, order, x_loc, u_loc, ws, n_total, p0):
        """Enqueue the fit of this rank's points [p0, p0 + P) with the fused gather (P may be 0)."""
        P = 0 if x_loc is None else x_loc.shape[0]
        prm, nprm = system._params()
        _lib.call("irs_smooth_finalize_gather", system.system_id, prm, nprm, order, _device.ptr(x_loc),
                  _device.ptr(u_loc), P, 1 if ws is None else ws.C, None if ws is None else _device.ptr(ws.partials),
                  self._hout.buffer_ptrs_dev, self._hflags.buffer_ptrs_dev, _device.ptr(self.epoch),
                  _device.ptr(self.counter), self.out_stride, int(p0), self.T, self.rank, self.world,
                  self.timeout_s, float(n_total), 0 if ws is None or not ws.centered else 1,
                  None if ws is None else _device.ptr(ws.ct), _device.stream_ptr())

    def step_done(self):
        """Count one executed step (eager or replayed from a graph) and return device views
        (At [T,n,n], Bt [T,n,m], ct [T,n], status [T] float64) of its full result: the parity half of the
        output buffer the kernels of that step wrote (valid once the stream has run them)."""
        self.calls += 1
        T, n, m = self.T, self.n, self.m
        o = self.out[(self.calls & 1) * self.out_stride:]
        na, nb, nc = T * n * n, T * n * m, T * n
        return (o[:na].view(T, n, n), o[na:na + nb].view(T, n, m), o[na + nb:na + nb + nc].view(T, n),
                o[na + nb + nc:na + nb + nc + T])

    def finalize(self, system, order, x_loc, u_loc, ws, n_total, p0):
        self.enqueue(system, order, x_loc, u_loc, ws, n_total, p0)
        return self.step_done()


def peer_capacity(system, order):
    """Nominal points per call the fused exchange supports (its blocks must be co-resident)."""
    import ctypes
    cap = ctypes.c_int(0)
    _lib.call("irs_smooth_finalize_peer_capacity", system.system_id, order, ctypes.byref(cap))
    return cap.value


class ShardedLinearizer:
    def __init__(self, system, order, group=None, peer_memory=None, peer_timeout_s=None):
        """peer_memory: None = use the fused peer-memory exchange when symmetric memory can be set up
        (NCCL all-gather otherwise), False = always NCCL, True = require it."""
        if getattr(system, "lib", _lib.MAIN) is not _lib.MAIN:
            raise NotImplementedError("sharded multi-GPU linearization is built for the library's own systems; "
                                      "a CudaSourceDynamics runs on one GPU")
        self.system, self.order, self.group = system, order, group
        self._ws = None
        self._peer_memory = peer_memory
        self._peer_timeout_s = peer_timeout_s
        self._px = None
        self._tg = None
        self._graphs = GraphRunner()

    def _workspace(self, P, N, fill=False):
        """fill: pick the chunk size so that the launch holds about 1.5 resident grids of work items (a rank's
        share of a strongly scaled step is small: with the default 4096-sample chunks 100 points x 12,500
        samples are 400 items for 740 block slots).  Only where bit-identity with the single-GPU run is not
        part of the contract (the sample axis: its summation order differs from one GPU's anyway)."""
        chunk = 0
        if fill and self.order == smoothing.ZERO_ORDER:
            C, _ = smoothing.plan(self.system.system_id, self.order, P, N)
            if P * C < 1100:
                chunk = max(512, -(-(N * P // 1100) // 256) * 256)
                if chunk >= 4096:
                    chunk = 0
        key = (self.system.system_id, self.order, P, N) if not chunk else (self.system.system_id, self.order, P, N, chunk)
        if self._ws is None or self._ws.key != key:
            self._ws = smoothing.Workspace(self.system, self.order, P, N, chunk)
        return self._ws

    def linearize_t(self, x_nom, u_nom, N, **kw):
        """Timestep-sharded.  x_nom [T,n], u_nom [T,m] replicated on every rank; returns the full
        (At, Bt, ct, status) on every rank — bit-identical to the single-GPU linearization (global point
        index in the Philox counter, per-point reduction order unchanged).  With peer memory the gather
        of the per-step blocks is fused into the fit kernel (TimestepGather: status is then a float64
        vector, 0 ok / 1 rank deficient / 2 a rank did not deliver); otherwise NCCL all-gather."""
        T = x_nom.shape[0]
        n, m = self.system.dim_x, self.system.dim_u
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        start, stop, _ = shard_range(T, world, rank)
        tg = self._timestep_gather(T)
        if tg is not None:
            p_base = kw.pop("p0", 0)
            ws = self._workspace(stop - start, N) if stop > start else None
            xs, us = (x_nom[start:stop], u_nom[start:stop]) if stop > start else (None, None)   # contiguous row slices

            def enqueue():
                if ws is not None:
                    smoothing.accumulate(self.system, self.order, xs, us, N, ws, p0=start + p_base, **kw)
                tg.enqueue(self.system, self.order, xs, us, ws, N, start)

            # two launches per step, replayed from a CUDA graph (the epoch of the gather lives on the device)
            key = None
            if kw.get("noise") is None and kw.get("sigma") is not None and ws is not None:
                key = (self.system.system_id, self.order, T, N, world, rank, kw.get("flags", 0), kw.get("stream_id", 0),
                       p_base, x_nom.data_ptr(), u_nom.data_ptr(), id(tg),
                       tuple(float(v) for v in self.system.device_params()))

            def update(handle):
                sig = np.ascontiguousarray(np.asarray(kw["sigma"], dtype=np.float32))
                _lib.call("irs_graph_update_smoothing", handle, sig.ctypes.data, int(kw.get("seed", 0)),
                          int(kw.get("it", 1)), int(kw.get("stream_id", 0)))

            self._graphs.run("linearize_t", key, enqueue, update)
            return tg.step_done()
        width = n * (n + m + 1) + 1
        if stop > start:
            ws = self._workspace(stop - start, N)
            xs, us = x_nom[start:stop].contiguous(), u_nom[start:stop].contiguous()
            smoothing.accumulate(self.system, self.order, xs, us, N, ws, p0=start, **kw)
            At, Bt, ct, status = smoothing.finalize(self.system, self.order, xs, us, ws, N)
            local = torch.cat((pack_abc(At, Bt, ct), status.to(torch.float64).unsqueeze(1)), dim=1)
        else:
            local = torch.zeros((0, width), dtype=torch.float64, device=x_nom.device)
        full = gather_rows(local, T, self.group)
        At, Bt, ct = unpack_abc(full[:, :width - 1], n, m)
        return At, Bt, ct, full[:, width - 1].to(torch.int32)

    def _timestep_gather(self, T):
        if self._peer_memory is False:
            return None
        if self._tg is None or self._tg.T != T:
            try:
                self._tg = TimestepGather(self.system, T, self.group, self._peer_timeout_s)
            except Exception as e:      # no symmetric memory on this system: NCCL (plumbing only)
                if self._peer_memory is True:
                    raise
                self._peer_memory = False
                self._tg = None
                import warnings
                warnings.warn("peer-memory gather unavailable (%s); using NCCL all-gather" % e)
        return self._tg

    def _peer_exchange(self, P, width):
        """The fused exchange for P points per call, or None (NCCL all-gather path).  An exchange is
        re-created (collectively: every rank sees the same P) only when P outgrows it; a SMALLER P
        reuses it — flags are per point and the epoch lives on the device, so nothing can go stale."""
        if self._peer_memory is False:
            return None
        if P > peer_capacity(self.system, self.order):
            if self._peer_memory is True:
                raise RuntimeError("the fused peer exchange needs all %d finalize blocks co-resident" % P)
            return None
        if self._px is None or not self._px.fits(P, width):
            try:
                self._px = PeerExchange(P, width, self.group, self._peer_timeout_s)
                self._graphs.reset()        # captured sequences point at the old exchange
            except Exception as e:      # no symmetric memory on this system: fall back to NCCL (plumbing only)
                if self._peer_memory is True:
                    raise
                self._peer_memory = False
                self._px = None
                import warnings
                warnings.warn("peer-memory exchange unavailable (%s); using NCCL all-gather" % e)
        return self._px

    def linearize_n_numpy(self, x_trj, u_trj, N_local, **kw):
        """linearize_n with numpy in / numpy out — the sample-sharded counterpart of
        IrsLqrZeroOrder.get_TV_matrices: one pinned host->device copy of [x_nom | u_nom], the kernels
        and the exchange, one device->host copy of [At | Bt | ct | status]; returns
        (At, Bt, ct, status) fitted on all W * N_local samples, identical on every rank.  Raises
        (smoothing.check_status) on a rank-deficient fit or a peer-exchange timeout."""
        T = min(np.asarray(u_trj).shape[0], np.asarray(x_trj).shape[0])
        ws = self._workspace(T, N_local, fill=True)
        ws.stage_nominal(x_trj, u_trj)
        ws.enqueue_upload()
        self.linearize_n(ws.x_nom, ws.u_nom, N_local, **kw)      # the fit lands in ws.At / Bt / ct / status
        ws.enqueue_download()
        At, Bt, ct, status = ws.read_download()
        smoothing.check_status(status)
        return At, Bt, ct, status

    def linearize_n(self, x_nom, u_nom, N_local, **kw):
        """Sample-sharded.  Every rank draws N_local samples per point (global sample index
        rank*N_local + i); returns (At, Bt, ct, status) fitted on all W*N_local samples.  No host
        synchronisation: a failed exchange shows up as status 2 (smoothing.check_status raises).
        With in-kernel noise and the fused exchange the two launches of a step (accumulate, finalize with
        the exchange inside) are replayed from a CUDA graph from the third call of a shape on — the epoch
        of the exchange lives in device memory, only seed / iteration / sigma are re-parameterised."""
        T = x_nom.shape[0]
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if kw.get("flags", 0) & 8 and kw.get("noise") is None and N_local % 2 and world > 1:
            raise ValueError("antithetic pairs must not straddle ranks: N_local must be even (got %d)" % N_local)
        ws = self._workspace(T, N_local, fill=True)
        px = self._peer_exchange(T, ws.width)

        def enqueue():
            smoothing.accumulate(self.system, self.order, x_nom, u_nom, N_local, ws, i0=rank * N_local, **kw)
            if px is not None:
                px.finalize(self.system, self.order, x_nom, u_nom, ws, world * N_local)
            else:
                mine = smoothing.reduce_chunks(self.system, self.order, ws)
                everyone = gather_ranks(mine, self.group)
                smoothing.finalize(self.system, self.order, x_nom, u_nom, ws, world * N_local,
                                   reduced=everyone, nranks=world, rank_stride=mine.numel())

        key = None
        if px is not None and kw.get("noise") is None and kw.get("sigma") is not None:
            # everything a captured kernel reads besides (seed, it, sigma) must be part of the key
            key = (self.system.system_id, self.order, T, N_local, world, rank, kw.get("flags", 0),
                   kw.get("stream_id", 0), kw.get("p0", 0), x_nom.data_ptr(), u_nom.data_ptr(), id(px), ws.S,
                   tuple(float(v) for v in self.system.device_params()))

        def update(handle):
            sig = np.ascontiguousarray(np.asarray(kw["sigma"], dtype=np.float32))
            _lib.call("irs_graph_update_smoothing", handle, sig.ctypes.data, int(kw.get("seed", 0)),
                      int(kw.get("it", 1)), int(kw.get("stream_id", 0)))

        self._graphs.run("linearize_n", key, enqueue, update)
        return ws.At, ws.Bt, ws.ct, ws.status
