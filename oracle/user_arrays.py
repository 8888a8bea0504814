"""TEST INFRASTRUCTURE ONLY — user-written systems that read arrays (CudaSourceDynamics(arrays=...)) and their
float64 twins.

- A linear plant x' = A x + B u + c of any (n, m): `linear_arrays` draws A, B, c from a seed, `LINEAR_STEP` reads
  them as arrays and `linear_literal_step` writes the same numbers into the body as literals.
- A Linear-act-Linear-act-Linear network x' = net([x, u]) (`MLP_STEP`, activation ReLU through fmax), or a
  cart-pole-shaped residual model x' = x + h (g(x, u) + net([x, u])) with g = [v, w, u, -u] (`RESIDUAL_MLP_STEP`,
  activation tanh), weights W1 b1 W2 b2 W3 b3 in torch.nn.Linear layout, and `MlpTwin`, both in float64 numpy.
- A cart on a line whose thrust is a piecewise-linear curve of its speed, read from a table at the index
  floor((v - v0) / dv) (`THRUST_STEP`, `ThrustTwin`).
"""
import numpy as np

LINEAR_STEP = """
    for (int i = 0; i < A_n0; ++i) {
        R acc = c[i];
        for (int j = 0; j < A_n1; ++j) acc += A(i, j) * x[j];
        for (int k = 0; k < Bu_n1; ++k) acc += Bu(i, k) * u[k];
        o[i] = acc;
    }
"""


def linear_arrays(n, m, seed=0):
    rng = np.random.default_rng(seed)
    return {"A": 0.95 * np.eye(n) + 0.03 * rng.standard_normal((n, n)), "Bu": 0.2 * rng.standard_normal((n, m)),
            "c": 0.01 * rng.standard_normal(n)}


def linear_literal_step(arrays):
    """LINEAR_STEP with the coefficients as literals (%.17g: the same doubles; float rounds them once, as the
    fp32 copy of an array does)."""
    A, B, c = arrays["A"], arrays["Bu"], arrays["c"]
    n, m = B.shape
    lines = []
    for i in range(n):
        terms = ["R(%.17g)" % c[i]] + ["R(%.17g) * x[%d]" % (A[i, j], j) for j in range(n)] + \
                ["R(%.17g) * u[%d]" % (B[i, k], k) for k in range(m)]
        lines.append("    {\n        R acc = %s;\n%s        o[%d] = acc;\n    }" % (
            terms[0], "".join("        acc += %s;\n" % t for t in terms[1:]), i))
    return "\n".join(lines) + "\n"


class LinearTwin:
    def __init__(self, arrays):
        self.A, self.B, self.c = arrays["A"], arrays["Bu"], arrays["c"]
        self.dim_x, self.dim_u = self.B.shape
        self.h = 0.0

    def dynamics_batch(self, x, u):
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        return x @ self.A.T + u @ self.B.T + self.c

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]

    def jacobian_xu_batch(self, x, u):
        J = np.hstack((self.A, self.B))
        return np.broadcast_to(J, (np.atleast_2d(x).shape[0],) + J.shape).copy()

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(x, u)[0]


_MLP_BODY = """
    R a1[W1_n0];
#pragma unroll
    for (int j = 0; j < W1_n0; ++j) {
        R s = b1[j];
#pragma unroll
        for (int k = 0; k < N; ++k) s += W1(j, k) * x[k];
#pragma unroll
        for (int k = 0; k < M; ++k) s += W1(j, N + k) * u[k];
        a1[j] = %(act1)s;
    }
    R acc[W3_n0];
#pragma unroll
    for (int i = 0; i < W3_n0; ++i) acc[i] = b3[i];
    for (int j = 0; j < W2_n0; ++j) {
        R s = b2[j];
#pragma unroll
        for (int k = 0; k < W2_n1; ++k) s += W2(j, k) * a1[k];
        const R a = %(act2)s;
#pragma unroll
        for (int i = 0; i < W3_n0; ++i) acc[i] += W3(i, j) * a;
    }
%(out)s
"""
MLP_STEP = _MLP_BODY % dict(act1="fmax(s, R(0))", act2="fmax(s, R(0))", out="""#pragma unroll
    for (int i = 0; i < N; ++i) o[i] = acc[i];""")
RESIDUAL_MLP_STEP = _MLP_BODY % dict(act1="tanh(s)", act2="tanh(s)", out="""    o[0] = x[0] + h * (x[2] + acc[0]);
    o[1] = x[1] + h * (x[3] + acc[1]);
    o[2] = x[2] + h * (u[0] + acc[2]);
    o[3] = x[3] + h * (acc[3] - u[0]);""")


def residual_drive(x, u):
    """g(x, u) of RESIDUAL_MLP_STEP; works on numpy arrays and torch tensors [B, .]."""
    return [x[:, 2], x[:, 3], u[:, 0], -u[:, 0]]


def mlp_arrays(weights):
    W1, b1, W2, b2, W3, b3 = weights
    return {"W1": W1, "b1": b1, "W2": W2, "b2": b2, "W3": W3, "b3": b3}


class MlpTwin:
    """The network of MLP_STEP (relu) or RESIDUAL_MLP_STEP (tanh, h) in float64."""

    def __init__(self, weights, dim_x, dim_u, act="relu", h=0.0):
        self.W1, self.b1, self.W2, self.b2, self.W3, self.b3 = [np.asarray(w, dtype=np.float64) for w in weights]
        self.dim_x, self.dim_u, self.h, self.act = dim_x, dim_u, h, act

    def dynamics_batch(self, x, u):
        xu = np.hstack((np.atleast_2d(x), np.atleast_2d(u)))
        f = (lambda a: np.maximum(a, 0.0)) if self.act == "relu" else np.tanh
        out = f(f(xu @ self.W1.T + self.b1) @ self.W2.T + self.b2) @ self.W3.T + self.b3
        if self.act == "relu":
            return out
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        return x + self.h * (np.stack(residual_drive(x, u), 1) + out)

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]


def cartpole_net(seed=0, hidden=64):
    """A 5-64-64-4 tanh network built with torch on the CPU from a seed -> (torch module in float64, weights)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    layers = [torch.nn.Linear(5, hidden), torch.nn.Tanh(), torch.nn.Linear(hidden, hidden), torch.nn.Tanh(),
              torch.nn.Linear(hidden, 4)]
    with torch.no_grad():
        for mod in layers:
            if isinstance(mod, torch.nn.Linear):
                bound = 1.0 / np.sqrt(mod.in_features)
                mod.weight.copy_(torch.empty_like(mod.weight).uniform_(-bound, bound, generator=g))
                mod.bias.copy_(torch.empty_like(mod.bias).uniform_(-bound, bound, generator=g))
    net = torch.nn.Sequential(*layers).double()
    weights = []
    for mod in layers:
        if isinstance(mod, torch.nn.Linear):
            weights += [mod.weight.detach().numpy().copy(), mod.bias.detach().numpy().copy()]
    return net, weights


# x = [position, speed], u = [throttle]; p = [drag, v0, 1 / dv]; thrust(v) interpolates tab between
# v0 + k dv and v0 + (k + 1) dv, clamped to the table's ends
THRUST_STEP = """
    const R drag = p[0], v0 = p[1], idv = p[2];
    const R s = (x[1] - v0) * idv;
    int k = (int)floor(s);
    k = k < 0 ? 0 : (k > tab_n0 - 2 ? tab_n0 - 2 : k);
    const R fr = s - R(k);
    const R lo = tab[k], hi = tab[k + 1];
    const R thrust = lo + fr * (hi - lo);
    o[0] = x[0] + h * x[1];
    o[1] = x[1] + h * (thrust * u[0] - drag * x[1]);
"""
THRUST_PARAMS = [0.3, -3.0, 2.0]            # drag, v0, 1 / dv: the table spans v in [-3, 3] in steps of 0.5
THRUST_H = 0.05


def thrust_table():
    v = np.linspace(-3.0, 3.0, 13)
    return 2.0 - 0.15 * v * v + 0.1 * np.sin(3.0 * v)


class ThrustTwin:
    def __init__(self, tab, h=THRUST_H, params=THRUST_PARAMS):
        self.tab, self.h = np.asarray(tab, dtype=np.float64), h
        self.drag, self.v0, self.idv = params
        self.dim_x, self.dim_u = 2, 1

    def dynamics_batch(self, x, u):
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        s = (x[:, 1] - self.v0) * self.idv
        k = np.clip(np.floor(s).astype(np.int64), 0, self.tab.size - 2)
        fr = s - k
        thrust = self.tab[k] + fr * (self.tab[k + 1] - self.tab[k])
        return np.stack((x[:, 0] + self.h * x[:, 1], x[:, 1] + self.h * (thrust * u[:, 0] - self.drag * x[:, 1])), 1)

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]
