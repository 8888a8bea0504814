"""Host driver of the randomized-smoothing linearization kernels.

`linearize(...)` is the device-level entry: nominal points already on the GPU in, (At, Bt, ct) on
the GPU out, no host synchronisation.  It implements the numeric core of
IrsLqrZeroOrder.get_TV_matrices (irs_lqr/irs_lqr_zero_order.py:38-63) and
IrsLqrFirstOrder.get_TV_matrices (irs_lqr/irs_lqr_first_order.py:28-54) for all nominal points at
once; the per-timestep Python loop of the reference becomes the grid's y-extent.
"""
import ctypes

import numpy as np
import torch

from . import _device, _lib

ZERO_ORDER = 0
FIRST_ORDER = 1
# smoothing flags (include/irs_mpc_b200.h)
FLAG_PROJECT_ABSOLUTE, FLAG_PROJECT_DELTA, FLAG_ANTITHETIC, FLAG_CENTERED = 2, 4, 8, 16


def plan(system_id, order, P, N, chunk_samples=0, lib=_lib.MAIN):
    """(C, S): C chunks of S samples per nominal point; chunk_samples = 0 is the library default."""
    C = ctypes.c_int(0)
    S = ctypes.c_longlong(0)
    lib.call("irs_smooth_plan", system_id, order, P, N, int(chunk_samples), ctypes.byref(C), ctypes.byref(S))
    return C.value, S.value


class Workspace:
    """Reusable device buffers for one (system, order, P, N) shape.

    The fit outputs live in ONE flat float64 buffer [At | Bt | ct | status(int32)] and the nominal
    points in one [x_nom | u_nom] buffer, each with a pinned host mirror, so that the numpy-facing
    API moves exactly one host->device and one device->host copy per linearization."""

    def __init__(self, system, order, P, N, chunk_samples=0):
        self.key = (system.system_key, order, P, N) if not chunk_samples else (system.system_key, order, P, N, chunk_samples)
        self.C, self.S = plan(system.system_id, order, P, N, chunk_samples, lib=system.lib)
        self.width = system.lib.handle().irs_partial_width(system.system_id, order)
        n, m = system.dim_x, system.dim_u
        self.P, self.n, self.m = P, n, m
        self.partials = _device.empty((P, self.C, self.width), torch.float32)
        na, nb, nc = P * n * n, P * n * m, P * n
        self._out = _device.empty((na + nb + nc + (P + 1) // 2,))
        self.At = self._out[:na].view(P, n, n)
        self.Bt = self._out[na:na + nb].view(P, n, m)
        self.ct = self._out[na + nb:na + nb + nc].view(P, n)
        self.status = self._out[na + nb + nc:].view(torch.int32)[:P]
        self._nom = _device.empty((P * (n + m),))
        self.x_nom = self._nom[:P * n].view(P, n)
        self.u_nom = self._nom[P * n:].view(P, m)
        self._out_host = None
        self._nom_host = None
        # the last accumulate into this workspace was centred (regressors relative to the nominal point +
        # first moments: three_cart absolute points): the finalize must undo the shift
        self.centered = False

    def _host_buffers(self):
        if self._nom_host is None:
            self._nom_host = torch.empty(self._nom.shape, dtype=torch.float64).pin_memory()
            self._out_host = torch.empty(self._out.shape, dtype=torch.float64).pin_memory()
            self._nom_host_np = self._nom_host.numpy()      # numpy views of the pinned mirrors
            self._out_host_np = self._out_host.numpy()

    def stage_nominal(self, x_trj, u_trj):
        """numpy [>=P, n], [>=P, m] -> the pinned host mirror of [x_nom | u_nom] (no device work)."""
        P, n, m = self.P, self.n, self.m
        self._host_buffers()
        h = self._nom_host_np
        h[:P * n] = np.asarray(x_trj, dtype=np.float64)[:P].reshape(-1)
        h[P * n:] = np.asarray(u_trj, dtype=np.float64)[:P].reshape(-1)

    def enqueue_upload(self):
        self._host_buffers()
        self._nom.copy_(self._nom_host, non_blocking=True)

    def enqueue_download(self):
        self._host_buffers()
        self._out_host.copy_(self._out, non_blocking=True)

    def read_download(self):
        """Synchronise and unpack the pinned mirror -> (At, Bt, ct, status) numpy arrays."""
        P, n, m = self.P, self.n, self.m
        torch.cuda.current_stream().synchronize()
        h = self._out_host_np.copy()      # ONE copy out of the pinned mirror; the results are views of it
        na, nb, nc = P * n * n, P * n * m, P * n
        At = h[:na].reshape(P, n, n)
        Bt = h[na:na + nb].reshape(P, n, m)
        ct = h[na + nb:na + nb + nc].reshape(P, n)
        status = h[na + nb + nc:].view(np.int32)[:P]
        return At, Bt, ct, status

    def h2d_bytes(self):
        return self._nom.numel() * 8

    def d2h_bytes(self):
        return self._out.numel() * 8


def accumulate(system, order, x_nom, u_nom, N, ws, sigma=None, noise=None, seed=0, it=1,
               stream_id=0, p0=0, i0=0, flags=0, point_range=None):
    """Launch the accumulation kernel: partial Gram blocks (order 0) or Jacobian sums (order 1).
    point_range = (lo, hi): only the nominal points lo..hi-1 of (x_nom, u_nom, ws) — the Philox
    counters carry the global point index, so the ranges of a split launch reproduce the full one."""
    partials = ws.partials
    if point_range is not None:
        lo, hi = point_range
        x_nom, u_nom, partials = x_nom[lo:hi], u_nom[lo:hi], partials[lo:hi]
        noise = None if noise is None else noise[lo:hi]
        p0 += lo
    P = x_nom.shape[0]
    prm, nprm = system._params()
    if system.batch_differs_from_scalar and order == ZERO_ORDER:
        flags |= 1   # IRS_SAMPLES_BATCH_VARIANT: samples go through dynamics_batch (…zero_order.py:51)
    ws.centered = order == ZERO_ORDER and bool(flags & (FLAG_PROJECT_ABSOLUTE | FLAG_CENTERED))
    sig = None
    if noise is None:
        sig = np.ascontiguousarray(np.asarray(sigma, dtype=np.float32))
        if sig.shape != (system.dim_x + system.dim_u,):
            raise ValueError("sigma must have n + m = %d entries" % (system.dim_x + system.dim_u))
        sig = sig.ctypes.data_as(ctypes.c_void_p)
    fn = ("irs_smooth_zero_order_accumulate" if order == ZERO_ORDER
          else "irs_smooth_first_order_accumulate")
    system.lib.call(fn, system.system_id, prm, nprm, flags, _device.ptr(x_nom), _device.ptr(u_nom), P,
              int(N), sig, _device.ptr(noise), int(seed), int(it), int(stream_id),
              int(p0), int(i0), ws.C, ws.S, _device.ptr(partials), _device.stream_ptr())


def reduce_chunks(system, order, ws, out=None):
    """[P, C, width] fp32 partials -> [P, width] fp64 (the block exchanged between ranks)."""
    P = ws.partials.shape[0]
    if out is None:
        out = _device.empty((P, ws.width))
    system.lib.call("irs_smooth_reduce_chunks", system.system_id, order, _device.ptr(ws.partials), P, ws.C,
              _device.ptr(out), _device.stream_ptr())
    return out


def finalize(system, order, x_nom, u_nom, ws, n_total, partials=None, reduced=None, nranks=1,
             rank_stride=0, point_range=None):
    """Fit from fp32 per-chunk partials (default: ws.partials) or from fp64 reduced blocks.
    point_range = (lo, hi): only the nominal points lo..hi-1 (single-rank partials only)."""
    prm, nprm = system._params()
    part = None if reduced is not None else (ws.partials if partials is None else partials)
    At, Bt, ct, status = ws.At, ws.Bt, ws.ct, ws.status
    if point_range is not None:
        lo, hi = point_range
        assert reduced is None and nranks == 1
        x_nom, u_nom, part = x_nom[lo:hi], u_nom[lo:hi], part[lo:hi]
        At, Bt, ct, status = At[lo:hi], Bt[lo:hi], ct[lo:hi], status[lo:hi]
    P = x_nom.shape[0]
    system.lib.call("irs_smooth_finalize", system.system_id, prm, nprm, order, _device.ptr(x_nom),
              _device.ptr(u_nom), P, ws.C, _device.ptr(part), _device.ptr(reduced), nranks,
              int(rank_stride), float(n_total), 1 if ws.centered else 0, _device.ptr(At), _device.ptr(Bt),
              _device.ptr(ct), _device.ptr(status), _device.stream_ptr())
    return ws.At, ws.Bt, ws.ct, ws.status


def linearize(system, order, x_nom, u_nom, N, ws=None, **kw):
    """x_nom [P,n], u_nom [P,m] (CUDA float64) -> (At, Bt, ct, status) CUDA tensors."""
    P = x_nom.shape[0]
    if ws is None or ws.key != (system.system_key, order, P, N):
        ws = Workspace(system, order, P, N)
    accumulate(system, order, x_nom, u_nom, N, ws, **kw)
    return finalize(system, order, x_nom, u_nom, ws, N) + (ws,)


def check_status(status):
    """status per nominal point: 0 ok, 1 rank-deficient fit, 2 peer exchange timed out (multi-GPU)."""
    if isinstance(status, torch.Tensor):
        status = status.detach().cpu().numpy()
    status = np.asarray(status)
    if not status.any():
        return
    late = int(np.count_nonzero(status == 2))
    if late:
        raise RuntimeError(
            "peer exchange timed out: the Gram blocks of %d nominal point(s) did not arrive from every rank "
            "(a rank is missing, far behind, or issued a different call sequence); the fit was NOT computed"
            % late)
    bad = int(np.count_nonzero(status))
    raise np.linalg.LinAlgError(
        "smoothing fit: the sample Gram matrix [dx du]^T[dx du] is rank deficient at %d "
        "nominal point(s) (too few samples, NaN in the dynamics, or regressors whose offset dwarfs "
        "their spread — three_cart's projection='absolute' quirk far from the origin: the Gram is "
        "accumulated in fp32)" % bad)
