"""DynamicalSystem plug-in contract (mirrors irs_lqr/dynamical_system.py:1-66 of the reference).

The base class keeps the reference's attributes (`h`, `dim_x`, `dim_u`) and four virtual methods.
`CudaDynamicalSystem` is the base of the four built-in analytic systems: it carries the id and
parameter vector of the `__device__` functor compiled into libirs_mpc_b200.so and implements the
four methods by launching the batched kernels (numpy float64 in, numpy float64 out).
"""
import numpy as np
import torch

from . import _device, _lib


class DynamicalSystem:
    def __init__(self):
        self.h = 0
        self.dim_x = 0
        self.dim_u = 0

    def dynamics(self, x, u):
        """x (n,), u (m,) -> next state (n,)."""
        raise NotImplementedError("This class is virtual.")

    def dynamics_batch(self, x, u):
        """x (B, n), u (B, m) -> next states (B, n)."""
        raise NotImplementedError("This class is virtual.")

    def jacobian_xu(self, x, u):
        """-> (n, n+m): first n columns df/dx, last m columns df/du."""
        raise NotImplementedError("This class is virtual.")

    def jacobian_xu_batch(self, x, u):
        """-> (B, n, n+m)."""
        raise NotImplementedError("This class is virtual.")


class CudaDynamicalSystem(DynamicalSystem):
    """A system whose dynamics exist as a CUDA functor (system_id) inside the extension."""

    system_id = -1
    system_name = ""
    batch_differs_from_scalar = False   # only three_cart (SURVEY Appendix A-4)
    lib = _lib.MAIN                     # the library holding the functor (user systems: their own)
    riccati_segments = True             # the library has the segmented Riccati kernel for (dim_x, dim_u)

    @property
    def system_key(self):
        """Tells systems apart in workspace and CUDA-graph cache keys (user systems all have one id)."""
        return self.system_id

    def device_params(self):
        """Parameter vector in the order documented in include/irs_mpc_b200.h."""
        raise NotImplementedError

    # -- helpers ------------------------------------------------------------------------------
    def _params(self):
        return _lib.params_array(self.device_params())

    def _run_dynamics(self, x, u, batch_variant, dtype=torch.float64):
        x = np.asarray(x)
        u = np.asarray(u)
        if x.ndim != 2 or u.ndim != 2 or x.shape[1] != self.dim_x or u.shape[1] != self.dim_u \
                or x.shape[0] != u.shape[0]:
            raise ValueError("expected x (B,%d) and u (B,%d), got %s and %s"
                             % (self.dim_x, self.dim_u, x.shape, u.shape))
        B = x.shape[0]
        xd = _device.to_device(x, dtype)
        ud = _device.to_device(u, dtype)
        out = _device.empty((B, self.dim_x), dtype)
        prm, nprm = self._params()
        fn = "irs_dynamics_batch_f64" if dtype == torch.float64 else "irs_dynamics_batch_f32"
        self.lib.call(fn, self.system_id, prm, nprm, int(batch_variant), _device.ptr(xd),
                  _device.ptr(ud), _device.ptr(out), B, _device.stream_ptr())
        return _device.to_numpy(out).astype(np.float64)

    # -- DynamicalSystem API ------------------------------------------------------------------
    def dynamics(self, x, u):
        return self._run_dynamics(np.asarray(x)[None, :], np.asarray(u)[None, :], False)[0]

    def dynamics_batch(self, x, u):
        return self._run_dynamics(x, u, True)

    def jacobian_xu_batch(self, x, u, dtype=torch.float64):
        x = np.asarray(x)
        u = np.asarray(u)
        if x.ndim != 2 or u.ndim != 2 or x.shape[1] != self.dim_x or u.shape[1] != self.dim_u \
                or x.shape[0] != u.shape[0]:
            raise ValueError("expected x (B,%d) and u (B,%d), got %s and %s"
                             % (self.dim_x, self.dim_u, x.shape, u.shape))
        B = x.shape[0]
        xd = _device.to_device(x, dtype)
        ud = _device.to_device(u, dtype)
        J = _device.empty((B, self.dim_x, self.dim_x + self.dim_u), dtype)
        prm, nprm = self._params()
        fn = "irs_jacobian_xu_batch_f64" if dtype == torch.float64 else "irs_jacobian_xu_batch_f32"
        self.lib.call(fn, self.system_id, prm, nprm, _device.ptr(xd), _device.ptr(ud), _device.ptr(J),
                  B, _device.stream_ptr())
        return _device.to_numpy(J).astype(np.float64)

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None, :], np.asarray(u)[None, :])[0]
