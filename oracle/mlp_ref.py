"""TEST INFRASTRUCTURE ONLY — restatement of the reference's learned dynamics.

examples/pendulum/pendulum_nn.py:19-33 defines the network (Linear(3, 100) ReLU Linear(100, 100) ReLU
Linear(100, 2)), :66-90 wraps it as a DynamicalSystem:
  dynamics / dynamics_batch (:72-81)  x+ = net(float32([x, u])) -> numpy (float32 values)
  jacobian_xu (:83-90)                torch.autograd.grad of each output w.r.t. the input: the exact
                                      derivative of the piecewise-linear network.
Restated here in numpy with float32 arithmetic (the module's dtype); `dtype=np.float64` gives the float64 twin of
the same network (weights and inputs taken as given, every operation in float64) that the fp32 kernels are
bounded against at other hidden widths (tests/test_mlp_widths_kernels.py).  Pinned against torch itself — the
reference's evaluator — on the fixture written by oracle/make_mlp_fixture.py (tests/golden/mlp_pendulum.npz:
torch forward outputs and autograd Jacobians of a network trained the way pendulum_nn.py:35-62 trains it).
Only tests/, smoke() and bench.py's CPU legs may import this module.
"""
import numpy as np


class MlpOracle:
    def __init__(self, weights, dim_x=2, dim_u=1, h=0.0, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        self.W1, self.b1, self.W2, self.b2, self.W3, self.b3 = [np.asarray(w, dtype=self.dtype) for w in weights]
        self.dim_x, self.dim_u, self.h = dim_x, dim_u, h

    def _hidden(self, xu):
        xu = np.asarray(xu, dtype=self.dtype)                     # torch.Tensor(...) in pendulum_nn.py:73,78
        zero = self.dtype.type(0)
        a1 = np.maximum(xu @ self.W1.T + self.b1, zero)
        a2 = np.maximum(a1 @ self.W2.T + self.b2, zero)
        return a1, a2

    def dynamics_batch(self, x, u):
        # pendulum_nn.py:77-81
        _, a2 = self._hidden(np.hstack((np.asarray(x), np.asarray(u))))
        return (a2 @ self.W3.T + self.b3).astype(np.float64)

    def dynamics(self, x, u):
        # pendulum_nn.py:72-76
        return self.dynamics_batch(np.asarray(x)[None], np.asarray(u)[None])[0]

    def jacobian_xu_batch(self, x, u, masks=None):
        # pendulum_nn.py:83-90 for every row: d out / d in = W3 diag(a2 > 0) W2 diag(a1 > 0) W1
        # masks: (a1 > 0 [B, H1], a2 > 0 [B, H2]) taken from another evaluation (the float32 activations of a
        # kernel) in place of this oracle's own
        if masks is None:
            a1, a2 = self._hidden(np.hstack((np.asarray(x), np.asarray(u))))
            masks = (a1 > 0, a2 > 0)
        m1 = np.asarray(masks[0]).astype(self.dtype)
        m2 = np.asarray(masks[1]).astype(self.dtype)
        r2 = self.W3[None, :, :] * m2[:, None, :]                 # [B, n, H2]
        r1 = (r2 @ self.W2) * m1[:, None, :]                      # [B, n, H1]
        return (r1 @ self.W1).astype(np.float64)                  # [B, n, d]

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(np.asarray(x)[None], np.asarray(u)[None])[0]
