"""Sampling objects for the smoothing kernels.

The reference takes `sampling(xbar, ubar, iter) -> (dx[N,n], du[N,m])`, a Python closure drawing
from numpy's global RNG (irs_lqr/irs_lqr_zero_order.py:12-22; e.g.
examples/pendulum/pendulum_zero_order.py:38-43).  Any such callable is still honoured (it is
called T times and the result replayed through the kernels).  `GaussianSampling` describes the
same distribution declaratively so that the noise can be generated inside the kernel with
Philox4x32-7 and never touches HBM:

    sigma_iter = sigma0 / iter**power          (variance stepping of the example scripts)
    delta[i, c] = sigma_iter[c] * normal(seed; sample i, point t, iter, stream)

It is also callable with the reference signature, in which case it returns exactly the deltas
the fused kernel would draw for that (t, iter) — generated on the GPU by irs_philox_dump.
"""
import ctypes

import numpy as np
import torch

from . import _device, _lib

PROJECTION_MODES = (None, "absolute", "delta")


class GaussianSampling:
    def __init__(self, sigma_x, sigma_u, num_samples, power=0.5, seed=0x1255, projection=None,
                 stream_id=0, antithetic=True):
        """projection: None | "absolute" (reference quirk, three_cart_zero_order.py:43 returns
        projection(...) = absolute points) | "delta" (corrected: projected point minus nominal).
        antithetic: draw the samples in pairs x +- z (sample 2q = +z_q, 2q+1 = -z_q).  Every sample
        keeps the marginal N(0, sigma^2) of the reference's closure; the even-order terms of the dynamics
        cancel exactly in the fit, and the fused kernel draws one Philox / Box-Muller block and stages
        one Gram row per pair.  False: independent samples as in the reference's `np.random.normal`."""
        if projection not in PROJECTION_MODES:
            raise ValueError("projection must be one of %s" % (PROJECTION_MODES,))
        self.sigma0 = np.concatenate((np.atleast_1d(np.asarray(sigma_x, dtype=np.float64)),
                                      np.atleast_1d(np.asarray(sigma_u, dtype=np.float64))))
        self.dim_x = np.atleast_1d(sigma_x).shape[0]
        self.dim_u = np.atleast_1d(sigma_u).shape[0]
        self.num_samples = int(num_samples)
        self.power = float(power)
        self.seed = int(seed)
        self.projection = projection
        self.stream_id = int(stream_id)
        self.antithetic = bool(antithetic)
        self._t = 0   # timestep counter used when called through the reference closure signature

    def sigma(self, it):
        return self.sigma0 / (float(it) ** self.power)

    def sigma32(self, it):
        """sigma(it) as the contiguous float32 array (and its pointer) the kernels take; the last
        iteration's array is kept (the schedule is a pure function of `it`)."""
        c = getattr(self, "_sigma32_cache", None)
        if c is None or c[0] != it:
            arr = np.ascontiguousarray(self.sigma(it), dtype=np.float32)
            c = (it, arr, arr.ctypes.data_as(ctypes.c_void_p))
            self._sigma32_cache = c
        return c[1], c[2]

    def flags(self):
        return {None: 0, "absolute": 2, "delta": 4}[self.projection] | (8 if self.antithetic else 0)

    def deltas(self, T, it, t0=0, i0=0, num_samples=None, return_words=False):
        """Deltas [T, N, d] (numpy float32) exactly as the fused kernels draw them."""
        N = self.num_samples if num_samples is None else int(num_samples)
        d = self.sigma0.shape[0]
        sig = np.ascontiguousarray(self.sigma(it), dtype=np.float32)
        out = _device.empty((T, N, d), torch.float32)
        words = _device.empty((T, N, (d + 3) // 4, 4), torch.int32) if return_words else None
        _lib.call("irs_philox_dump", T, N, d, sig.ctypes.data_as(ctypes.c_void_p), self.seed, int(it), self.stream_id,
                  int(t0), int(i0), 1 if self.antithetic else 0, _device.ptr(words), _device.ptr(out),
                  _device.stream_ptr())
        z = _device.to_numpy(out)
        if return_words:
            return z, _device.to_numpy(words).view(np.uint32)
        return z

    def reset_timestep(self):
        self._t = 0

    def __call__(self, xbar, ubar, it):
        """Reference closure signature.  Successive calls within one iteration walk t = 0, 1, ...
        (get_TV_matrices calls sampling once per timestep in order, irs_lqr_zero_order.py:49-50)."""
        if it != getattr(self, "_t_iter", None):      # a new iteration starts again at t = 0
            self._t, self._t_iter = 0, it
        z = self.deltas(1, it, t0=self._t)[0].astype(np.float64)
        self._t += 1
        return z[:, :self.dim_x], z[:, self.dim_x:]


def project_samples(system, x, dx, u, du):
    """three_cart_dynamics.py:196-264 on the GPU: absolute (x + dx projected, u + du)."""
    x_abs = np.asarray(x, dtype=np.float64) + np.asarray(dx, dtype=np.float64)
    u_abs = np.asarray(u, dtype=np.float64) + np.asarray(du, dtype=np.float64)
    xd = _device.to_device(x_abs, torch.float64)
    prm, nprm = system._params()
    system.lib.call("irs_project_batch_f64", system.system_id, prm, nprm, _device.ptr(xd), xd.shape[0],
              _device.stream_ptr())
    return _device.to_numpy(xd), u_abs
