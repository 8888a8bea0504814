"""User-written dynamics (CudaSourceDynamics): CUDA C++ bodies compiled into a library of their own.

Test systems are source strings below with float64 numpy twins.  The pendulum and bicycle bodies are those of
csrc/systems.cuh, so every kernel they reach is the built-in system's kernel with the same functor arithmetic:
their results are compared bit for bit with the built-in systems.  The cart-pole (4, 1) and a 3-D double
integrator with drag (6, 3: nine regressors, not a built-in pair) are compared with the float64 oracle on the
kernel's own deltas at the bars of test_gpu_parity.py.
"""
import concurrent.futures
import ctypes

import numpy as np
import pytest

from irs_mpc_b200 import _lib, user_system
from oracle import cpu_restatement as cr
from oracle import example_configs as ec

PENDULUM_STEP = """
    R s, c;
    Math<R>::sincos(x[0], s, c);
    const R v = x[1] + h * (u[0] - s);
    o[1] = v;
    o[0] = x[0] + h * v;
"""
PENDULUM_JAC = """
    R s, c;
    Math<R>::sincos(x[0], s, c);
    J[0] = R(1) - h * h * c;  J[1] = h;     J[2] = h * h;
    J[3] = -h * c;            J[4] = R(1);  J[5] = h;
"""
DAMPED_PENDULUM_STEP = """
    R s, c;
    Math<R>::sincos(x[0], s, c);
    const R v = x[1] + h * (u[0] - s - p[0] * x[1]);
    o[1] = v;
    o[0] = x[0] + h * v;
"""
BICYCLE_STEP = """
    R s, c, sd, cd;
    Math<R>::sincos(x[2], s, c);
    Math<R>::sincos(x[4], sd, cd);
    const R v = x[3];
    o[0] = x[0] + h * (v * c);
    o[1] = x[1] + h * (v * s);
    o[2] = x[2] + h * (v * Math<R>::div(sd, cd));
    o[3] = x[3] + h * u[0];
    o[4] = x[4] + h * u[1];
"""
BICYCLE_JAC = """
    R s, c, sd, cd;
    Math<R>::sincos(x[2], s, c);
    Math<R>::sincos(x[4], sd, cd);
    const R icd = Math<R>::rcp(cd);
    for (int i = 0; i < N * D; ++i) J[i] = R(0);
    for (int i = 0; i < N; ++i) J[i * D + i] = R(1);
    J[0 * D + 2] = -h * (x[3] * s);
    J[0 * D + 3] = h * c;
    J[1 * D + 2] = h * (x[3] * c);
    J[1 * D + 3] = h * s;
    J[2 * D + 3] = h * (sd * icd);
    J[2 * D + 4] = h * (x[3] * icd * icd);
    J[3 * D + 5] = h;
    J[4 * D + 6] = h;
"""
# cart-pole: x = [cart position, pole angle, cart velocity, pole rate], u = [force]; p = [mc, mp, l, g]
CARTPOLE_STEP = """
    const R mc = p[0], mp = p[1], l = p[2], g = p[3];
    R s, c;
    Math<R>::sincos(x[1], s, c);
    const R den = mc + mp * s * s;
    const R w2 = x[3] * x[3];
    const R xdd = (u[0] + mp * s * (l * w2 + g * c)) / den;
    const R thdd = (-u[0] * c - mp * l * w2 * c * s - (mc + mp) * g * s) / (l * den);
    o[0] = x[0] + h * x[2];
    o[1] = x[1] + h * x[3];
    o[2] = x[2] + h * xdd;
    o[3] = x[3] + h * thdd;
"""
CARTPOLE_JAC = """
    const R mc = p[0], mp = p[1], l = p[2], g = p[3];
    R s, c;
    Math<R>::sincos(x[1], s, c);
    const R den = mc + mp * s * s, dden = R(2) * mp * s * c;
    const R w = x[3], w2 = w * w;
    const R xdd = (u[0] + mp * s * (l * w2 + g * c)) / den;
    const R thdd = (-u[0] * c - mp * l * w2 * c * s - (mc + mp) * g * s) / (l * den);
    const R dxdd_th = (mp * (c * (l * w2 + g * c) - g * s * s) - xdd * dden) / den;
    const R dthdd_th = (u[0] * s - mp * l * w2 * (c * c - s * s) - (mc + mp) * g * c - thdd * l * dden) / (l * den);
    for (int i = 0; i < N * D; ++i) J[i] = R(0);
    for (int i = 0; i < N; ++i) J[i * D + i] = R(1);
    J[0 * D + 2] = h;
    J[1 * D + 3] = h;
    J[2 * D + 1] = h * dxdd_th;
    J[2 * D + 3] = h * (R(2) * mp * l * w * s / den);
    J[2 * D + 4] = h / den;
    J[3 * D + 1] = h * dthdd_th;
    J[3 * D + 3] = R(1) + h * (-R(2) * mp * w * c * s / den);
    J[3 * D + 4] = h * (-c / (l * den));
"""
# 3-D double integrator with speed-dependent drag: x = [position (3), velocity (3)], u = acceleration; p = [drag]
DRAG_STEP = """
    const R sp = sqrt(R(1) + x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
    for (int i = 0; i < 3; ++i) {
        const R v = x[3 + i] + h * (u[i] - p[0] * x[3 + i] * sp);
        o[3 + i] = v;
        o[i] = x[i] + h * v;
    }
"""
CARTPOLE_PARAMS = [1.0, 0.1, 0.5, 9.81]

# name -> (dim_x, dim_u, h, params, step, jacobian)
SPECS = {
    "pendulum_src": (2, 1, 0.05, [], PENDULUM_STEP, PENDULUM_JAC),
    "damped_pendulum": (2, 1, 0.05, [0.3], DAMPED_PENDULUM_STEP, None),
    "bicycle_src": (5, 2, 0.1, [], BICYCLE_STEP, BICYCLE_JAC),
    "cartpole": (4, 1, 0.02, CARTPOLE_PARAMS, CARTPOLE_STEP, CARTPOLE_JAC),
    "cartpole_nojac": (4, 1, 0.02, CARTPOLE_PARAMS, CARTPOLE_STEP, None),
    "drag3d": (6, 3, 0.05, [0.2], DRAG_STEP, None),
}


class CartPoleOracle:
    def __init__(self, h, params=CARTPOLE_PARAMS):
        self.h, (self.mc, self.mp, self.l, self.g) = h, params
        self.dim_x, self.dim_u = 4, 1

    def dynamics_batch(self, x, u):
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        mc, mp, l, g, h = self.mc, self.mp, self.l, self.g, self.h
        s, c = np.sin(x[:, 1]), np.cos(x[:, 1])
        den = mc + mp * s * s
        w2 = x[:, 3] * x[:, 3]
        xdd = (u[:, 0] + mp * s * (l * w2 + g * c)) / den
        thdd = (-u[:, 0] * c - mp * l * w2 * c * s - (mc + mp) * g * s) / (l * den)
        return np.stack([x[:, 0] + h * x[:, 2], x[:, 1] + h * x[:, 3], x[:, 2] + h * xdd, x[:, 3] + h * thdd], 1)

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]

    def jacobian_xu_batch(self, x, u, eps=1e-6):
        xu = np.hstack((np.atleast_2d(x), np.atleast_2d(u)))
        J = np.zeros((xu.shape[0], 4, 5))
        for j in range(5):
            e = np.zeros(5)
            e[j] = eps
            J[:, :, j] = (self.dynamics_batch((xu + e)[:, :4], (xu + e)[:, 4:]) -
                          self.dynamics_batch((xu - e)[:, :4], (xu - e)[:, 4:])) / (2 * eps)
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(x, u)[0]


class DragOracle:
    def __init__(self, h, drag=0.2):
        self.h, self.drag = h, drag
        self.dim_x, self.dim_u = 6, 3

    def dynamics_batch(self, x, u):
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        sp = np.sqrt(1.0 + np.sum(x[:, 3:] ** 2, axis=1, keepdims=True))
        v = x[:, 3:] + self.h * (u - self.drag * x[:, 3:] * sp)
        return np.hstack((x[:, :3] + self.h * v, v))

    def dynamics(self, x, u):
        return self.dynamics_batch(x, u)[0]


def cartpole_cfg(T):
    return dict(h=0.02, T=T, Q=np.diag([1.0, 10.0, 0.1, 0.1]), Qd=np.diag([100.0, 100.0, 10.0, 10.0]),
                R=np.diag([0.1]), x0=np.zeros(4), xd_trj=np.tile([0.0, np.pi, 0.0, 0.0], (T + 1, 1)),
                u_trj_initial=np.tile([0.5], (T, 1)), sigma=np.array([0.05, 0.1, 0.2, 0.3, 1.0]))


def drag_cfg(T):
    return dict(h=0.05, T=T, Q=np.diag([1.0, 1, 1, 0.1, 0.1, 0.1]), Qd=np.diag([50.0, 50, 50, 5, 5, 5]),
                R=np.diag([0.1, 0.1, 0.1]), x0=np.zeros(6), xd_trj=np.tile([1.0, -1.0, 0.5, 0, 0, 0], (T + 1, 1)),
                u_trj_initial=np.tile([0.1, 0.0, -0.1], (T, 1)), sigma=np.array([0.05] * 3 + [0.1] * 3 + [0.5] * 3))


@pytest.fixture(scope="module")
def built():
    """Every test system's library, compiled once (in parallel) -> name: (path, seconds, hash)."""
    with concurrent.futures.ThreadPoolExecutor(len(SPECS)) as pool:
        futs = {name: pool.submit(user_system.build_library, n, m, 1 + len(prm), step, jac, name)
                for name, (n, m, h, prm, step, jac) in SPECS.items()}
        return {name: f.result() for name, f in futs.items()}


_SYSTEMS = {}


def system(built, name):
    if name not in _SYSTEMS:
        n, m, h, prm, step, jac = SPECS[name]
        _SYSTEMS[name] = user_system.CudaSourceDynamics(n, m, h, prm, step=step, jacobian=jac, name=name)
    return _SYSTEMS[name]


def params_of(api, cfg, T=None):
    p = api.IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial"):
        setattr(p, key, cfg[key])
    for key in ("xbound", "ubound"):
        setattr(p, key, cfg.get(key))
    return p


@pytest.fixture(scope="module")
def api():
    import irs_mpc_b200.all as a
    return a


# ------------------------------------------------------------------------------------------------
# CPU: validation, build, cache, ABI
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kw,match", [
    (dict(dim_x=12, dim_u=5), "16"),
    (dict(params=[1.0] * 10), "at most 9"),
    (dict(params=[1.0, float("nan")]), "finite"),
    (dict(h=float("inf")), "finite"),
    (dict(dim_x=0), "positive"),
])
def test_limits_are_checked_before_compiling(monkeypatch, kw, match):
    monkeypatch.setattr(user_system, "_compile", lambda *a: pytest.fail("compiled"))
    args = dict(dim_x=2, dim_u=1, h=0.05, params=[], step=PENDULUM_STEP)
    args.update(kw)
    with pytest.raises(ValueError, match=match):
        user_system.CudaSourceDynamics(**args)


def test_compile_error_points_into_the_body(tmp_path, monkeypatch):
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    bad = "R s, c;\nMath<R>::sincos(x[0], s, c);\no[0] = x[0] + h * s\no[1] = x[1];\n"
    with pytest.raises(RuntimeError, match=r"step\(4\)"):      # the missing ';' shows at the next line
        user_system.build_library(2, 1, 1, bad, None, "broken")


def test_cache_hit_runs_no_compiler(built, monkeypatch):
    def refuse(*a):
        raise AssertionError("the compiler ran")
    monkeypatch.setattr(user_system, "_compile", refuse)
    n, m, h, prm, step, jac = SPECS["cartpole_nojac"]
    s = user_system.CudaSourceDynamics(n, m, h, prm, step=step, name="cartpole_nojac")
    assert s.cache_hit and s.library_path == built["cartpole_nojac"][0]


def test_no_compiler_uses_the_cache_or_says_so(built, monkeypatch):
    monkeypatch.setattr(user_system, "_nvcc_version", lambda nvcc: None)
    n, m, h, prm, step, jac = SPECS["drag3d"]
    path, seconds, _ = user_system.build_library(n, m, 1 + len(prm), step, jac, "drag3d")
    assert path == built["drag3d"][0] and seconds == 0.0
    with pytest.raises(RuntimeError, match="no CUDA compiler"):
        user_system.build_library(n, m, 1 + len(prm), step + "\n// another system", jac, "drag3d")


@pytest.mark.parametrize("name", sorted(SPECS))
def test_library_loads_and_reports_its_system(built, name):
    n, m = SPECS[name][:2]
    lib = _lib.Library.at(built[name][0])
    h = lib.handle()                        # dlopen + signature table + ABI check
    assert h.irs_abi_version() == _lib.ABI_VERSION
    dims = [ctypes.c_int() for _ in range(3)]
    lib.call("irs_system_dims", user_system.USER_SYSTEM_ID, *[ctypes.byref(v) for v in dims])
    d = n + m
    assert [v.value for v in dims] == [n, m, n * d]
    assert h.irs_partial_width(user_system.USER_SYSTEM_ID, 0) == d * (d + 1) // 2 + d * n
    assert h.irs_partial_width(user_system.USER_SYSTEM_ID, 1) == n * d
    assert h.irs_system_dims(6, None, None, None) != 0          # one system id past the table


def test_without_jacobian_the_jacobian_paths_refuse(built, api):
    s = system(built, "cartpole_nojac")
    assert not s.has_jacobian
    with pytest.raises(NotImplementedError):
        s.jacobian_xu(np.zeros(4), np.zeros(1))
    cfg = cartpole_cfg(10)
    with pytest.raises(NotImplementedError):
        api.IrsLqrExact(s, params_of(api, cfg))
    with pytest.raises(NotImplementedError):
        api.IrsLqrFirstOrder(s, params_of(api, cfg), api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 100))


def test_sharded_paths_refuse_user_systems(built):
    from irs_mpc_b200.distributed import ShardedLinearizer
    with pytest.raises(NotImplementedError):
        ShardedLinearizer(system(built, "drag3d"), 0)


def test_systems_keep_apart_in_cache_keys(built):
    a, b = system(built, "damped_pendulum"), system(built, "cartpole_nojac")
    assert a.system_id == b.system_id and a.system_key != b.system_key and a.lib is not b.lib
    assert len({v[2] for v in built.values()}) == len(built)        # one source hash per system


# ------------------------------------------------------------------------------------------------
# GPU: the built-in systems' twins, bit for bit
# ------------------------------------------------------------------------------------------------
TWINS = [("pendulum_src", "PendulumDynamics", ec.pendulum), ("bicycle_src", "BicycleDynamics", ec.bicycle)]


def twin_pair(built, api, name, cls):
    s = system(built, name)
    return s, getattr(api, cls)(s.h)


@pytest.mark.gpu
@pytest.mark.parametrize("name,cls,cfgf", TWINS)
def test_twin_dynamics_bit_identical(built, api, name, cls, cfgf):
    import torch
    s, b = twin_pair(built, api, name, cls)
    rng = np.random.default_rng(3)
    x, u = rng.standard_normal((4096, s.dim_x)), rng.standard_normal((4096, s.dim_u))
    for dt in (torch.float32, torch.float64):
        assert np.array_equal(s._run_dynamics(x, u, True, dt), b._run_dynamics(x, u, True, dt))
    assert np.array_equal(s.dynamics(x[0], u[0]), b.dynamics(x[0], u[0]))
    assert np.array_equal(s.dynamics_batch(x, u), b.dynamics_batch(x, u))
    # the Jacobian body writes J directly; the built-in assembles it from the varying scalars: same products
    np.testing.assert_allclose(s.jacobian_xu_batch(x, u), b.jacobian_xu_batch(x, u), rtol=0, atol=1e-15)


@pytest.mark.gpu
@pytest.mark.parametrize("name,cls,cfgf", TWINS)
@pytest.mark.parametrize("engine", [0, 1])
def test_twin_zero_order_and_descent_bit_identical(built, api, name, cls, cfgf, engine):
    T = 40
    cfg = cfgf(T=T)
    cfg["xbound"] = cfg["ubound"] = None      # the bounded descent has a test of its own
    s, b = twin_pair(built, api, name, cls)
    n = s.dim_x
    try:
        for lib in (s.lib, _lib.MAIN):
            lib.call("irs_set_gram_engine", engine)
        res = []
        for sysm in (s, b):
            sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], 3000, seed=5)
            solver = api.IrsLqrZeroOrder(sysm, params_of(api, cfg), sampler)
            lin = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
            rng = np.random.default_rng(9)

            def closure(x, u, it):
                return (rng.standard_normal((500, n)) * cfg["sigma"][:n],
                        rng.standard_normal((500, sysm.dim_u)) * cfg["sigma"][n:])
            replay = api.IrsLqrZeroOrder(sysm, params_of(api, cfg), closure)
            lin_r = replay.get_TV_matrices(replay.x_trj, replay.u_trj)
            xd, ud = solver.local_descent(solver.x_trj, solver.u_trj)
            x, u, c = solver.iterate(2, verbose=False)
            res.append(lin + lin_r + (xd, ud, np.array(solver.cost_lst), x, u))
    finally:
        for lib in (s.lib, _lib.MAIN):
            lib.call("irs_set_gram_engine", -1)
    for i, (a, bb) in enumerate(zip(*res)):
        assert np.array_equal(a, bb), (i, float(np.max(np.abs(a - bb))), float(np.max(np.abs(bb))))


@pytest.mark.gpu
@pytest.mark.parametrize("name,cls,cfgf", TWINS)
def test_twin_first_order_within_last_bits(built, api, name, cls, cfgf):
    """The user functor averages J; the built-in averages the varying scalars and assembles once (affine):
    the same sums up to the products h * v taken before or after the mean — a few ulp of J."""
    T = 30
    cfg = cfgf(T=T)
    s, b = twin_pair(built, api, name, cls)
    n = s.dim_x
    out = []
    for sysm in (s, b):
        sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], 4000, seed=2)
        solver = api.IrsLqrFirstOrder(sysm, params_of(api, cfg), sampler)
        out.append(solver.get_TV_matrices(solver.x_trj, solver.u_trj))
    for a, bb in zip(*out):
        np.testing.assert_allclose(a, bb, rtol=0, atol=1e-6 * max(1.0, float(np.abs(bb).max())))


@pytest.mark.gpu
def test_bicycle_active_steer_bound_bit_identical(built, api):
    T = 30
    cfg = ec.bicycle(T=T)
    cfg["ubound"] = np.array([[-1e4, -0.05], [1e4, 0.05]])       # the steer rate bound is active
    s, b = twin_pair(built, api, "bicycle_src", "BicycleDynamics")
    out = []
    for sysm in (s, b):
        sampler = api.GaussianSampling(cfg["sigma"][:5], cfg["sigma"][5:], 3000, seed=4)
        solver = api.IrsLqrZeroOrder(sysm, params_of(api, cfg), sampler)
        x, u = solver.local_descent(solver.x_trj, solver.u_trj)
        assert getattr(solver, "bounded_admm_iterations", 0) > 0
        assert np.all(np.abs(u[:, 1]) <= 0.05 + 1e-6)
        out.append((x, u))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


@pytest.mark.gpu
def test_twin_batched_instances_bit_identical(built, api):
    T, I = 30, 8
    cfg = ec.pendulum(T=T)
    s, b = twin_pair(built, api, "pendulum_src", "PendulumDynamics")
    x0 = np.random.default_rng(1).standard_normal((I, 2)) * 0.3
    out = []
    for sysm in (s, b):
        sampler = api.GaussianSampling(cfg["sigma"][:2], cfg["sigma"][2:], 2000, seed=3)
        bat = api.BatchedIrsLqrZeroOrder(sysm, cfg["Q"], cfg["Qd"], cfg["R"], x0, cfg["xd_trj"],
                                         cfg["u_trj_initial"], sampler)
        out.append(bat.iterate(2))
    for a, bb in zip(*out):
        assert np.array_equal(a, bb)


# ------------------------------------------------------------------------------------------------
# GPU: cart-pole and the (6, 3) system against the float64 oracle on the kernel's own deltas
# ------------------------------------------------------------------------------------------------
def rel(a, b):
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30))


ORACLE_CASES = [("cartpole", cartpole_cfg, CartPoleOracle), ("drag3d", drag_cfg, DragOracle)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfgf,oracle", ORACLE_CASES)
def test_zero_order_descent_against_oracle(built, api, name, cfgf, oracle):
    T, N = 30, 4000
    cfg = cfgf(T)
    s = system(built, name)
    n = s.dim_x
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, seed=7)
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler)
    orc = oracle(cfg["h"])
    x_o = cr.rollout(orc, cfg["x0"], cfg["u_trj_initial"])
    assert rel(solver.x_trj, x_o) < 1e-12
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    At_o, Bt_o, ct_o = cr.zero_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    assert rel(At, At_o) < 1e-4 and rel(Bt, Bt_o) < 1e-4 and float(np.max(np.abs(ct - ct_o))) < 1e-4
    x_new, u_new = solver.local_descent(solver.x_trj, solver.u_trj)
    # teacher-forced: the oracle's Riccati pass and rollout on the kernel's linearization
    K, k = cr.tvlqr_riccati(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["xd_trj"])
    x_t, u_t = cr.closed_loop_descent(orc, K, k, solver.x_trj[0])
    assert rel(x_new, x_t) < 1e-4 and rel(u_new, u_t) < 1e-4
    cost = solver.evaluate_cost(x_new, u_new)
    assert abs(cost - cr.evaluate_cost(x_t, u_t, cfg["xd_trj"], cfg["Q"], cfg["R"])) < 1e-4 * abs(cost)
    x_c, u_c = x_new + 0.0, u_new + 0.0               # new arrays: evaluate_cost runs its kernel
    c_dev = solver.evaluate_cost(x_c, u_c)
    c_o = cr.evaluate_cost(x_c, u_c, cfg["xd_trj"], cfg["Q"], cfg["R"])
    assert abs(c_dev - c_o) <= 1e-12 * abs(c_o)
    solver.iterate(5, verbose=False)
    assert solver.cost_lst[-1] < solver.cost_lst[0]


@pytest.mark.gpu
def test_drag3d_engines(built, api):
    """d = 9: the tcgen05 Gram by default; its rows do not split evenly over four warps, so a forced
    CUDA-core engine is refused with a message."""
    T, cfg = 10, drag_cfg(10)
    s = system(built, "drag3d")
    sampler = api.GaussianSampling(cfg["sigma"][:6], cfg["sigma"][6:], 2000, seed=1)
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler)
    solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    try:
        s.lib.call("irs_set_gram_engine", 0)
        with pytest.raises(_lib.IrsCudaError, match="evenly"):
            solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    finally:
        s.lib.call("irs_set_gram_engine", -1)


@pytest.mark.gpu
def test_cartpole_first_order_and_exact_against_oracle(built, api):
    T, N = 30, 4000
    cfg = cartpole_cfg(T)
    s = system(built, "cartpole")
    orc = CartPoleOracle(cfg["h"])
    rng = np.random.default_rng(0)
    x, u = 0.5 * rng.standard_normal((64, 4)), rng.standard_normal((64, 1))
    np.testing.assert_allclose(s.jacobian_xu_batch(x, u), orc.jacobian_xu_batch(x, u), rtol=0, atol=1e-7)
    sampler = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], N, seed=3)
    solver = api.IrsLqrFirstOrder(s, params_of(api, cfg), sampler)
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    At_o, Bt_o, ct_o = cr.first_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    assert rel(At, At_o) < 1e-4 and rel(Bt, Bt_o) < 1e-4 and float(np.max(np.abs(ct - ct_o))) < 1e-4
    exact = api.IrsLqrExact(s, params_of(api, cfg))
    At, Bt, ct = exact.get_TV_matrices(exact.x_trj, exact.u_trj)
    At_o, Bt_o, ct_o = cr.exact_tv_matrices(orc, exact.x_trj, exact.u_trj)
    assert rel(At, At_o) < 1e-7 and rel(Bt, Bt_o) < 1e-7 and float(np.max(np.abs(ct - ct_o))) < 1e-7 * max(1.0, float(np.abs(ct_o).max()))
    exact.iterate(3, verbose=False)
    assert exact.cost_lst[-1] < exact.cost_lst[0]


@pytest.mark.gpu
def test_wrong_jacobian_entry_is_refused(tmp_path, monkeypatch):
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    wrong = CARTPOLE_JAC.replace("J[2 * D + 4] = h / den;", "J[2 * D + 4] = -h / den;")
    assert wrong != CARTPOLE_JAC
    with pytest.raises(ValueError, match=r"J\[2\]\[4\]"):
        user_system.CudaSourceDynamics(4, 1, 0.02, CARTPOLE_PARAMS, step=CARTPOLE_STEP, jacobian=wrong, name="wrong")


@pytest.mark.gpu
def test_cartpole_bounded_descent_first_qp_is_certified(built, api):
    from oracle import box_kkt as bk
    from irs_mpc_b200 import _device
    from irs_mpc_b200.tv_lqr import box_solve_device
    T = 25
    cfg = cartpole_cfg(T)
    cfg["ubound"] = np.array([[-2.0], [2.0]])
    s = system(built, "cartpole")
    sampler = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 3000, seed=6)
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler)
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    big = 1e30 * np.ones(4)
    dev = [_device.to_device(v[None]) for v in (At, Bt, ct)]
    xq, uq, _, status, _ = box_solve_device(
        s, False, *dev, solver._dQ, solver._dQd, solver._dR, cfg["Q"], cfg["Qd"], cfg["R"], solver._dxd, 0,
        _device.to_device(cfg["x0"][None]), -big, big, np.array([-2.0]), np.array([2.0]))
    assert int(status.item()) == 0
    uq = _device.to_numpy(uq[0])
    qp = bk.BoxQP(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], -big, big,
                  np.array([-2.0]), np.array([2.0]))
    c = qp.certify(uq)
    assert c["certified"], (c["min_lam"], c["max_violation"], c["kkt_residual"])
    assert np.any(np.abs(np.abs(uq) - 2.0) < 1e-6)          # the bound is active
    # the bounded descent (box_mpc_kernel on the user functor) applies that QP's first input
    sampler2 = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 3000, seed=6)
    solver2 = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler2)
    x_new, u_new = solver2.local_descent(solver2.x_trj, solver2.u_trj)
    assert solver2.bounded_admm_iterations > 0
    assert abs(u_new[0, 0] - uq[0, 0]) < 1e-6 and np.all(np.abs(u_new) <= 2.0 + 1e-6)


@pytest.mark.gpu
def test_batched_shard_equals_unsharded(built, api):
    T, I = 25, 8
    cfg = cartpole_cfg(T)
    s = system(built, "cartpole")
    x0 = np.random.default_rng(2).standard_normal((I, 4)) * 0.1
    xd = np.broadcast_to(cfg["xd_trj"], (I, T + 1, 4)).copy()

    def run(lo, hi):
        sampler = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 2000, seed=8)
        bat = api.BatchedIrsLqrZeroOrder(s, cfg["Q"], cfg["Qd"], cfg["R"], x0[lo:hi], xd[lo:hi],
                                         cfg["u_trj_initial"], sampler, instance_offset=lo)
        return bat.iterate(2)
    full, part = run(0, I), run(3, 6)
    for a, b in zip(full, part):
        assert np.array_equal(a[3:6], b)


@pytest.mark.gpu
def test_cem_matches_numpy_restatement(built, api):
    T, B = 30, 128
    cfg = cartpole_cfg(T)
    s = system(built, "cartpole")
    p = api.CemParameters()
    p.Q, p.Qd, p.R, p.x0, p.xd_trj, p.u_trj_initial = (cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"],
                                                       cfg["u_trj_initial"])
    p.n_elite, p.batch_size, p.initial_std = 16, B, 0.5 * np.ones(1)
    np.random.seed(99)
    solver = api.CrossEntropyMethod(s, p)
    x_new, u_new = solver.local_descent(solver.x_trj, solver.u_trj)
    orc = CartPoleOracle(cfg["h"])
    np.random.seed(99)
    cand = np.random.normal(cfg["u_trj_initial"], np.tile(p.initial_std, (T, 1)), (B, T, 1))
    costs = np.array([cr.evaluate_cost(cr.rollout(orc, cfg["x0"], cand[k]), cand[k], cfg["xd_trj"], cfg["Q"],
                                       cfg["R"]) for k in range(B)])
    best = np.argpartition(costs, p.n_elite)[:p.n_elite]
    u_o = cand[best].mean(axis=0)
    np.testing.assert_allclose(u_new, u_o, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(x_new, cr.rollout(orc, cfg["x0"], u_o), rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
def test_graph_replay_equals_eager(built, api, monkeypatch):
    from irs_mpc_b200 import _graph
    T = 30
    cfg = cartpole_cfg(T)
    s = system(built, "cartpole")
    out = []
    for graphs in (True, False):
        monkeypatch.setattr(_graph, "USE_GRAPHS", graphs)
        sampler = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 3000, seed=12)
        solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler)
        res = [solver.local_descent(solver.x_trj, solver.u_trj) for _ in range(5)]     # replayed from the 3rd
        if graphs:
            assert solver._graphs._slots["descent"][1] is not None
        s.params = [1.2] + CARTPOLE_PARAMS[1:]          # a changed parameter re-captures
        res.append(solver.local_descent(solver.x_trj, solver.u_trj))
        res.append(solver.local_descent(solver.x_trj, solver.u_trj))
        res.append(solver.local_descent(solver.x_trj, solver.u_trj))
        s.params = list(CARTPOLE_PARAMS)
        out.append(res)
    for (xa, ua), (xb, ub) in zip(*out):
        assert np.array_equal(xa, xb) and np.array_equal(ua, ub)
    assert not np.array_equal(out[0][0][0], out[0][5][0])


@pytest.mark.gpu
def test_two_user_systems_share_nothing(built, api):
    """Same id, same dimensions, different dynamics: interleaved solvers give what each gives alone."""
    T = 30
    cfg = ec.pendulum(T=T)

    def make(name):
        sampler = api.GaussianSampling(cfg["sigma"][:2], cfg["sigma"][2:], 2000, seed=1)
        return api.IrsLqrZeroOrder(system(built, name), params_of(api, cfg), sampler)
    alone = []
    for name in ("pendulum_src", "damped_pendulum"):
        sv = make(name)
        alone.append([sv.local_descent(sv.x_trj, sv.u_trj) for _ in range(4)])
    a, b = make("pendulum_src"), make("damped_pendulum")
    mixed = [[], []]
    for _ in range(4):
        mixed[0].append(a.local_descent(a.x_trj, a.u_trj))
        mixed[1].append(b.local_descent(b.x_trj, b.u_trj))
    for i in range(2):
        for (xa, ua), (xb, ub) in zip(alone[i], mixed[i]):
            assert np.array_equal(xa, xb) and np.array_equal(ua, ub)
    assert not np.array_equal(alone[0][0][0], alone[1][0][0])
