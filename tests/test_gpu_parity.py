"""GPU parity tests (run with `-m gpu` on a B200).  Everything here calls the CUDA path through
the C ABI (ctypes) and compares with (a) vectors produced by the reference's own code
(tests/golden) and (b) the float64 oracle on identical inputs.

Tolerances: bit-exact for integer bookkeeping (Philox words, contact cases); 1e-4 relative
(max-abs error over max-abs value per array) for everything that passes through the fp32 sample
path, as stated in BASELINE.json:north_star; 1e-9 or tighter for the fp64 sequential kernels.
"""
import json
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import cpu_restatement as cr          # noqa: E402
from oracle import example_configs as ec          # noqa: E402
from oracle import philox_ref                     # noqa: E402

SYSTEMS = ["pendulum", "bicycle", "quadrotor", "three_cart"]
FP32_RTOL = 1e-4


def rel_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    import irs_mpc_b200.all as m
    return m


def make_system(api, name):
    cfg = ec.CONFIGS[name]()
    return api.__dict__[{"pendulum": "PendulumDynamics", "bicycle": "BicycleDynamics",
                         "quadrotor": "QuadrotorDynamics", "three_cart": "ThreeCartDynamics"}[name]](cfg["h"])


def make_params(api, cfg, T=None, x0=None, u_trj=None):
    p = api.IrsLqrParameters()
    T = cfg["T"] if T is None else T
    p.Q, p.Qd, p.R = cfg["Q"], cfg["Qd"], cfg["R"]
    p.x0 = cfg["x0"] if x0 is None else x0
    p.xd_trj = cfg["xd_trj"][:T + 1]
    p.u_trj_initial = cfg["u_trj_initial"][:T] if u_trj is None else u_trj
    p.xbound, p.ubound = cfg["xbound"], cfg["ubound"]
    return p


def gold(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


# ------------------------------------------------------------------------------------------------
# dynamics / jacobians / projection
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SYSTEMS)
def test_dynamics_fp64_matches_reference_vectors(api, golden_dir, name):
    g = gold(golden_dir, "dynamics_%s.npz" % name)
    s = make_system(api, name)
    fb = s.dynamics_batch(g["x"], g["u"])
    np.testing.assert_allclose(fb, g["f_batch"], rtol=0, atol=1e-12)
    fs = s._run_dynamics(g["x"], g["u"], False)
    np.testing.assert_allclose(fs, g["f_scalar"], rtol=0, atol=1e-12)
    one = s.dynamics(g["x"][3], g["u"][3])
    np.testing.assert_allclose(one, g["f_scalar"][3], rtol=0, atol=1e-12)


@pytest.mark.parametrize("name", SYSTEMS)
def test_dynamics_fp32_sample_path(api, golden_dir, name):
    import torch
    g = gold(golden_dir, "dynamics_%s.npz" % name)
    s = make_system(api, name)
    x32 = g["x"].astype(np.float32)
    u32 = g["u"].astype(np.float32)
    f32 = s._run_dynamics(x32, u32, True, dtype=torch.float32)
    orc = cr.SYSTEMS[name](s.h)
    ref = orc.dynamics_batch(x32.astype(np.float64), u32.astype(np.float64))
    if name == "three_cart":
        # fp32 rounding may flip a contact case for samples within one ulp of the threshold;
        # compare only rows whose float64 gaps are not marginal
        sfree = orc._free_step(x32.astype(np.float64), u32.astype(np.float64))
        margin = np.minimum(np.abs(sfree[:, 1] - sfree[:, 0] - 0.2), np.abs(sfree[:, 2] - sfree[:, 1] - 0.2))
        keep = margin > 1e-5
        assert keep.sum() > 0.95 * len(keep)
        f32, ref = f32[keep], ref[keep]
    assert rel_err(f32, ref) < 1e-5     # MUFU sin/cos/rcp approximations


def test_three_cart_contact_bookkeeping_bit_exact(api, golden_dir):
    """Which samples fall in which contact case is integer bookkeeping: the fp64 kernel must
    reproduce the oracle's case ids exactly (deduced from where batch and scalar semantics
    differ and from the velocity merge pattern)."""
    g = gold(golden_dir, "dynamics_three_cart.npz")
    s = make_system(api, "three_cart")
    orc = cr.ThreeCartOracle(s.h)
    case = orc.contact_case(g["x"], g["u"])
    fb = s._run_dynamics(g["x"], g["u"], True)
    fs = s._run_dynamics(g["x"], g["u"], False)
    free = orc._free_step(g["x"], g["u"])
    got = np.zeros_like(case)
    merged12 = (fb[:, 3] == fb[:, 4]) & (free[:, 3] != free[:, 4])
    merged23 = (fb[:, 4] == fb[:, 5]) & (free[:, 4] != free[:, 5])
    got[merged12 & merged23] = 1
    got[merged12 & ~merged23] = 2
    got[~merged12 & merged23] = 3
    np.testing.assert_array_equal(got, case)
    differs = np.any(fb != fs, axis=1)
    np.testing.assert_array_equal(differs, (case == 2) | (case == 3))


def test_three_cart_projection_matches_reference(api, golden_dir):
    g = gold(golden_dir, "dynamics_three_cart.npz")
    s = make_system(api, "three_cart")
    xp, up = s.projection(g["proj_xbar"], g["proj_dx"], g["proj_ubar"], g["proj_du"])
    np.testing.assert_allclose(xp, g["proj_x"], rtol=0, atol=1e-13)
    np.testing.assert_allclose(up, g["proj_u"], rtol=0, atol=1e-13)


@pytest.mark.parametrize("name", ["pendulum", "bicycle", "quadrotor"])
def test_jacobian_fp64_matches_oracle(api, golden_dir, name):
    g = gold(golden_dir, "dynamics_%s.npz" % name)
    s = make_system(api, name)
    orc = cr.SYSTEMS[name](s.h)
    J = s.jacobian_xu_batch(g["x"][:64], g["u"][:64])
    Jo = orc.jacobian_xu_batch(g["x"][:64], g["u"][:64])
    assert J.shape == Jo.shape
    assert rel_err(J, Jo) < 1e-11
    np.testing.assert_allclose(s.jacobian_xu(g["x"][0], g["u"][0]), Jo[0], rtol=0, atol=1e-9)


def test_three_cart_has_no_jacobian(api):
    s = make_system(api, "three_cart")
    with pytest.raises(NotImplementedError):
        s.jacobian_xu(np.zeros(6), np.zeros(2))


# ------------------------------------------------------------------------------------------------
# Philox bookkeeping
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("d", [3, 7, 8, 16])
def test_philox_words_bit_exact_and_normals(api, d, antithetic):
    sig = np.linspace(0.5, 2.0, d)
    s = api.GaussianSampling(sig[:d - 1], sig[d - 1:], 777, power=0.5, seed=0x1234ABCD5678, stream_id=5,
                             antithetic=antithetic)
    T, it, t0, i0 = 3, 4, 11, 1000
    z, words = s.deltas(T, it, t0=t0, i0=i0, return_words=True)
    ref_words = philox_ref.words_for(T, 777, d, s.seed, it, instance=5, t0=t0, i0=i0, antithetic=antithetic)
    np.testing.assert_array_equal(words, ref_words)
    ref_z = philox_ref.deltas(T, 777, s.sigma(it), s.seed, it, instance=5, t0=t0, i0=i0, antithetic=antithetic)
    np.testing.assert_allclose(z, ref_z, rtol=0, atol=2e-5 * float(np.max(s.sigma(it))))
    if antithetic:
        # index bookkeeping of the pairs is exact: sample 2q+1 is the bitwise negation of sample 2q
        # (i0 even), and an odd i0 starts on a - member
        np.testing.assert_array_equal(z[:, 1:777:2], -z[:, 0:776:2])
        np.testing.assert_array_equal(words[:, 1:777:2], words[:, 0:776:2])
        z_odd = s.deltas(T, it, t0=t0, i0=i0 + 1)
        np.testing.assert_array_equal(z_odd[:, :776], z[:, 1:])
    # the closure form walks timesteps in call order
    s.reset_timestep()
    dx0, du0 = s(None, None, it)
    dx1, du1 = s(None, None, it)
    z0 = s.deltas(2, it)
    np.testing.assert_array_equal(np.hstack((dx0, du0)).astype(np.float32), z0[0])
    np.testing.assert_array_equal(np.hstack((dx1, du1)).astype(np.float32), z0[1])


# ------------------------------------------------------------------------------------------------
# zero-order smoothing: replay against the REFERENCE's own outputs
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", SYSTEMS)
def test_zero_order_replay_matches_reference(api, golden_dir, name):
    g = gold(golden_dir, "zero_order_%s.npz" % name)
    cfg = ec.CONFIGS[name]()
    s = make_system(api, name)
    n = s.dim_x
    T = g["u_trj"].shape[0]
    deltas = g["deltas"]
    state = {"t": 0}

    def sampling(xbar, ubar, it):
        t = state["t"]
        state["t"] += 1
        dx = deltas[t][:, :n].astype(np.float64)
        du = deltas[t][:, n:].astype(np.float64)
        if cfg["projection"]:
            return s.projection(xbar, dx, ubar, du)     # as three_cart_zero_order.py:43
        return dx, du

    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=T, x0=g["x_trj"][0], u_trj=g["u_trj"]), sampling)
    np.testing.assert_allclose(solver.x_trj, g["x_trj"], rtol=0, atol=1e-12)
    assert abs(solver.cost - float(g["initial_cost"])) <= 1e-12 * abs(float(g["initial_cost"]))
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    assert At.shape == g["At"].shape and Bt.shape == g["Bt"].shape and ct.shape == g["ct"].shape
    assert rel_err(At, g["At"]) < FP32_RTOL
    assert rel_err(Bt, g["Bt"]) < FP32_RTOL
    assert rel_err(ct, g["ct"]) < FP32_RTOL


def test_zero_order_three_cart_inkernel_projection_matches_reference(api, golden_dir):
    """Same golden, but the projection runs inside the kernel (IRS_PROJECT_ABSOLUTE) on the raw
    deltas instead of in the Python closure."""
    import torch
    from irs_mpc_b200 import _device, smoothing
    g = gold(golden_dir, "zero_order_three_cart.npz")
    s = make_system(api, "three_cart")
    T = g["u_trj"].shape[0]
    x_nom = _device.to_device(g["x_trj"][:T])
    u_nom = _device.to_device(g["u_trj"])
    noise = _device.to_device(g["deltas"], torch.float32)
    At, Bt, ct, status, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x_nom, u_nom, noise.shape[1],
                                                noise=noise, flags=2)
    assert int(status.sum().item()) == 0
    assert rel_err(_device.to_numpy(At), g["At"]) < FP32_RTOL
    assert rel_err(_device.to_numpy(Bt), g["Bt"]) < FP32_RTOL
    assert rel_err(_device.to_numpy(ct), g["ct"]) < FP32_RTOL


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("name", SYSTEMS)
def test_zero_order_both_gram_engines_match_reference(api, golden_dir, name, engine):
    """CUDA-core (FFMA2) and tensor-core (tcgen05, bf16x2 split) Gram engines against the
    reference's own (At, Bt, ct) on the replayed deltas."""
    import torch
    from irs_mpc_b200 import _device, _lib, smoothing
    g = gold(golden_dir, "zero_order_%s.npz" % name)
    s = make_system(api, name)
    T = g["u_trj"].shape[0]
    x_nom = _device.to_device(g["x_trj"][:T])
    u_nom = _device.to_device(g["u_trj"])
    noise = _device.to_device(g["deltas"], torch.float32)
    _lib.call("irs_set_gram_engine", engine)
    try:
        At, Bt, ct, status, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x_nom, u_nom, noise.shape[1],
                                                    noise=noise, flags=2 if bool(g["projection"]) else 0)
        assert int(status.sum().item()) == 0
        At, Bt, ct = _device.to_numpy(At), _device.to_numpy(Bt), _device.to_numpy(ct)
    finally:
        _lib.call("irs_set_gram_engine", -1)
    scale = max(1.0, float(np.max(np.abs(g["x_trj"]))))
    assert rel_err(At, g["At"]) < FP32_RTOL
    assert rel_err(Bt, g["Bt"]) < FP32_RTOL
    assert float(np.max(np.abs(ct - g["ct"]))) < FP32_RTOL * scale


# ------------------------------------------------------------------------------------------------
# Philox fast path vs the oracle fed with the very same deltas
# ------------------------------------------------------------------------------------------------
def _nominal(api, name, T):
    cfg = ec.CONFIGS[name](T=T)
    s = make_system(api, name)
    rng = np.random.default_rng(42)
    u_trj = cfg["u_trj_initial"] + 0.05 * rng.standard_normal(cfg["u_trj_initial"].shape)
    return cfg, s, u_trj


@pytest.mark.parametrize("name,projection", [("pendulum", None), ("bicycle", None), ("quadrotor", None),
                                             ("three_cart", None), ("three_cart", "absolute"),
                                             ("three_cart", "delta")])
def test_zero_order_philox_matches_oracle_on_same_deltas(api, name, projection):
    T, N = 6, 3000
    cfg, s, u_trj = _nominal(api, name, T)
    n = s.dim_x
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=99,
                                   projection=projection)
    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=T, u_trj=u_trj), sampler)
    solver.iter = 3      # exercise the variance schedule sigma0 / iter**power
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    orc = cr.SYSTEMS[name](s.h)
    if projection is not None:
        for t in range(T):
            xp, up = orc.projection(solver.x_trj[t], deltas[t][:, :n], solver.u_trj[t], deltas[t][:, n:])
            if projection == "absolute":
                deltas[t] = np.hstack((xp, up))
            else:
                deltas[t][:, :n] = xp - solver.x_trj[t]
    At_o, Bt_o, ct_o = cr.zero_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    assert rel_err(At, At_o) < FP32_RTOL
    assert rel_err(Bt, Bt_o) < FP32_RTOL
    assert rel_err(ct, ct_o) < FP32_RTOL


@pytest.mark.parametrize("name", ["pendulum", "bicycle", "quadrotor"])
def test_first_order_philox_and_replay_match_oracle(api, name):
    T, N = 6, 2000
    cfg, s, u_trj = _nominal(api, name, T)
    n = s.dim_x
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=5)
    solver = api.IrsLqrFirstOrder(s, make_params(api, cfg, T=T, u_trj=u_trj), sampler)
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    orc = cr.SYSTEMS[name](s.h)
    At_o, Bt_o, ct_o = cr.first_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    assert rel_err(At, At_o) < FP32_RTOL
    assert rel_err(Bt, Bt_o) < FP32_RTOL
    assert rel_err(ct, ct_o) < FP32_RTOL
    # replay path through a plain closure returns the same thing
    sampler.reset_timestep()
    solver2 = api.IrsLqrFirstOrder(s, make_params(api, cfg, T=T, u_trj=u_trj),
                                   lambda xb, ub, it: sampler(xb, ub, it))
    At2, Bt2, ct2 = solver2.get_TV_matrices(solver2.x_trj, solver2.u_trj)
    assert rel_err(At2, At_o) < FP32_RTOL and rel_err(Bt2, Bt_o) < FP32_RTOL
    assert rel_err(ct2, ct_o) < FP32_RTOL


@pytest.mark.parametrize("name", ["pendulum", "bicycle", "quadrotor"])
def test_exact_matches_oracle(api, name):
    T = 7
    cfg, s, u_trj = _nominal(api, name, T)
    solver = api.IrsLqrExact(s, make_params(api, cfg, T=T, u_trj=u_trj))
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    orc = cr.SYSTEMS[name](s.h)
    At_o, Bt_o, ct_o = cr.exact_tv_matrices(orc, solver.x_trj, solver.u_trj)
    assert rel_err(At, At_o) < 1e-11 and rel_err(Bt, Bt_o) < 1e-11
    np.testing.assert_allclose(ct, ct_o, rtol=0, atol=1e-12 * max(1.0, float(np.max(np.abs(solver.x_trj)))))


# ------------------------------------------------------------------------------------------------
# TVLQR
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m", [(2, 1), (5, 2), (6, 2), (12, 4)])
def test_solve_tvlqr_matches_oracle(api, n, m):
    rng = np.random.default_rng(n * 10 + m)
    T = 25
    At = np.eye(n) + 0.1 * rng.standard_normal((T, n, n))
    Bt = 0.3 * rng.standard_normal((T, n, m))
    ct = 0.1 * rng.standard_normal((T, n))
    Q = np.diag(rng.uniform(0.5, 2.0, n))
    Qd = 10 * Q
    R = np.diag(rng.uniform(0.5, 2.0, m))
    x0 = rng.standard_normal(n)
    xd = rng.standard_normal((T + 1, n))
    xs, us = api.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd, api.get_solver("osqp"))
    xs_o, us_o = cr.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd)
    assert xs.shape == (T + 1, n) and us.shape == (T, m)
    assert rel_err(xs, xs_o) < 1e-9 and rel_err(us, us_o) < 1e-9


@pytest.mark.parametrize("I", [297, 1030])
def test_packed_riccati_for_many_instances_matches_oracle_and_block_kernel(api, I, monkeypatch):
    """For thousands of instances the quadrotor-sized backward pass runs two instances per warp with 4 x 4
    register tiles (tvlqr_riccati_packed_kernel; forced here below its switch point): gains against the float64 oracle (1e-9) and against the
    one-block-per-instance kernel (IRS_TVLQR_VARIANT=block; different summation order: 1e-10), instance
    counts that do not fill the last warp / block, per-instance desired trajectories, non-SPD steps flagged."""
    import torch
    from irs_mpc_b200 import _device
    from irs_mpc_b200.tv_lqr import riccati_device
    n, m, T = 12, 4, 9
    rng = np.random.default_rng(I)
    At = np.eye(n) + 0.1 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    Q = np.diag(rng.uniform(0.5, 2.0, n))
    Qd = 10 * Q + 0.3 * rng.standard_normal((n, n))
    Qd = Qd + Qd.T + 5 * np.eye(n)                             # dense, symmetric, positive definite
    R = np.diag(rng.uniform(0.5, 2.0, m))
    xd = rng.standard_normal((I, T + 1, n))
    dev = lambda v: _device.to_device(np.ascontiguousarray(v))
    args = (dev(At), dev(Bt), dev(ct), dev(Q), dev(Qd), dev(R), dev(xd), (T + 1) * n)
    monkeypatch.setenv("IRS_TVLQR_VARIANT", "packed")
    K, k, status = riccati_device(*args)
    assert int(status.sum().item()) == 0
    K, k = _device.to_numpy(K), _device.to_numpy(k)
    monkeypatch.setenv("IRS_TVLQR_VARIANT", "block")
    Kb, kb, sb = riccati_device(*args)
    monkeypatch.delenv("IRS_TVLQR_VARIANT", raising=False)
    assert rel_err(K, _device.to_numpy(Kb)) < 1e-10 and rel_err(k, _device.to_numpy(kb)) < 1e-10
    for b in (0, 1, 7, 8, I // 2, I - 2, I - 1):
        Ko, ko = cr.tvlqr_riccati(At[b], Bt[b], ct[b], Q, 0.5 * (Qd + Qd.T), R, xd[b])
        assert rel_err(K[b], Ko) < 1e-9 and rel_err(k[b], ko) < 1e-9, b
    # an indefinite terminal weight (H = R/2 + B'PB not SPD) is flagged for every instance
    monkeypatch.setenv("IRS_TVLQR_VARIANT", "packed")
    K2, k2, st2 = riccati_device(args[0], args[1], args[2], args[3], dev(-np.eye(n)), dev(1e-6 * R), args[6], args[7])
    monkeypatch.delenv("IRS_TVLQR_VARIANT", raising=False)
    assert int(st2.sum().item()) == I


def test_solve_tvlqr_error_conventions(api):
    n, m, T = 2, 1, 3
    At = np.tile(np.eye(n), (T, 1, 1))
    Bt = np.ones((T, n, m))
    ct = np.zeros((T, n))
    with pytest.raises(ValueError, match="TV_LQR failed"):
        api.solve_tvlqr(At, Bt, ct, -np.eye(n), -10 * np.eye(n), 1e-3 * np.eye(m), np.ones(n),
                        np.zeros((T + 1, n)), None)
    with pytest.raises(ValueError, match="Do not recognize solver"):
        api.get_solver("ipopt")


def test_constructor_error_conventions(api):
    cfg = ec.pendulum(T=10)
    s = make_system(api, "pendulum")
    p = make_params(api, cfg)
    p.Q = np.eye(3)
    with pytest.raises(RuntimeError, match="Q matrix"):
        api.IrsLqrExact(s, p)
    p = make_params(api, cfg)
    p.R = np.eye(2)
    with pytest.raises(RuntimeError, match="R matrix"):
        api.IrsLqrExact(s, p)
    empty = api.DynamicalSystem()
    with pytest.raises(RuntimeError, match="zero states"):
        api.IrsLqrExact(empty, make_params(api, cfg))

    class PyOnly(api.DynamicalSystem):
        def __init__(self):
            super().__init__()
            self.dim_x, self.dim_u = 2, 1

    with pytest.raises(RuntimeError, match="Could not evaluate dynamics"):
        api.IrsLqrExact(PyOnly(), make_params(api, cfg))


def test_rank_deficient_fit_raises(api):
    cfg = ec.quadrotor(T=3)
    s = make_system(api, "quadrotor")
    sampler = api.GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], 8, seed=1)   # N < d
    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=3), sampler)
    with pytest.raises(np.linalg.LinAlgError):
        solver.get_TV_matrices(solver.x_trj, solver.u_trj)


# ------------------------------------------------------------------------------------------------
# whole loop
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,key,rtol", [("pendulum", "pendulum_exact", 1e-10),
                                           ("quadrotor", "quadrotor_exact", 1e-7)])
def test_exact_loop_reproduces_stored_cost_curve(api, golden_dir, name, key, rtol):
    """examples/pendulum/analysis/pendulum_exact.csv and examples/quadrotor/analysis/
    quadrotor_exact.csv, free-running (no teacher forcing); the whole exact loop is fp64."""
    with open(os.path.join(golden_dir, "reference_costs.json")) as f:
        goldc = np.array(json.load(f)["stored_cost_curves"][key]["values"])
    cfg = ec.CONFIGS[name]()
    s = make_system(api, name)
    solver = api.IrsLqrExact(s, make_params(api, cfg))
    assert abs(solver.cost - goldc[0]) <= 1e-12 * goldc[0]
    solver.iterate(len(goldc) - 2, verbose=False)
    assert len(solver.cost_lst) == len(goldc)
    assert len(solver.x_trj_lst) == len(goldc) and len(solver.u_trj_lst) == len(goldc)
    np.testing.assert_allclose(np.array(solver.cost_lst), goldc, rtol=rtol)


@pytest.mark.parametrize("name,T,N", [("pendulum", 200, 1000), ("quadrotor", 40, 2000),
                                      ("three_cart", 30, 2000)])
def test_local_descent_teacher_forced_matches_oracle(api, name, T, N):
    """One descent from the same nominal trajectory with the same deltas: trajectory and cost
    within 1e-4 relative (BASELINE.json:north_star)."""
    cfg = ec.CONFIGS[name](T=T)
    s = make_system(api, name)
    n = s.dim_x
    proj = "absolute" if cfg["projection"] else None
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=2021,
                                   projection=proj)
    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=T), sampler)
    x_new, u_new = solver.local_descent(solver.x_trj, solver.u_trj)
    cost = solver.evaluate_cost(x_new, u_new)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    orc = cr.SYSTEMS[name](s.h)
    if proj:
        for t in range(T):
            xp, up = orc.projection(solver.x_trj[t], deltas[t][:, :n], solver.u_trj[t], deltas[t][:, n:])
            deltas[t] = np.hstack((xp, up))
    At, Bt, ct = cr.zero_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    K, k = cr.tvlqr_riccati(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["xd_trj"])
    x_o, u_o = cr.closed_loop_descent(orc, K, k, solver.x_trj[0])
    cost_o = cr.evaluate_cost(x_o, u_o, cfg["xd_trj"], cfg["Q"], cfg["R"])
    assert rel_err(x_new, x_o) < FP32_RTOL
    assert rel_err(u_new, u_o) < 5 * FP32_RTOL
    assert abs(cost - cost_o) / abs(cost_o) < FP32_RTOL
    assert abs(solver._last_descent_cost - cost) <= 1e-12 * abs(cost)


# ------------------------------------------------------------------------------------------------
# full-size, size-independent properties (BASELINE.json configs 3 and 4)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,N", [("quadrotor", 100000), ("three_cart", 200000)])
def test_full_size_properties(api, name, N):
    import torch
    from irs_mpc_b200 import _device, smoothing
    T = 100
    cfg = ec.CONFIGS[name](T=T)
    s = make_system(api, name)
    n = s.dim_x
    solver = api.IrsLqrExact(s, make_params(api, cfg, T=T)) if name != "three_cart" else None
    x_trj = cr.rollout(cr.SYSTEMS[name](s.h), cfg["x0"], cfg["u_trj_initial"])
    x_nom = _device.to_device(x_trj[:T])
    u_nom = _device.to_device(cfg["u_trj_initial"])
    kw = dict(sigma=cfg["sigma"], seed=0x1255, it=1)

    def run(xn, un, Ns, **extra):
        k = dict(kw)
        k.update(extra)
        At, Bt, ct, status, ws = smoothing.linearize(s, smoothing.ZERO_ORDER, xn, un, Ns, **k)
        assert int(status.sum().item()) == 0
        return At.clone(), Bt.clone(), ct.clone(), ws

    A1, B1, c1, ws = run(x_nom, u_nom, N)
    # (i) determinism: bit-identical on repeat
    A2, B2, c2, _ = run(x_nom, u_nom, N)
    assert torch.equal(A1, A2) and torch.equal(B1, B2) and torch.equal(c1, c2)
    # (ii) timestep sharding: computing the two halves of the horizon separately with the global
    #      point offset p0 reproduces the full result bit-for-bit (what the all-gather relies on)
    h = T // 2
    Aa, Ba, ca, _ = run(x_nom[:h].contiguous(), u_nom[:h].contiguous(), N, p0=0)
    Ab, Bb, cb, _ = run(x_nom[h:].contiguous(), u_nom[h:].contiguous(), N, p0=h)
    assert torch.equal(torch.cat((Aa, Ab)), A1) and torch.equal(torch.cat((Ba, Bb)), B1)
    assert torch.equal(torch.cat((ca, cb)), c1)
    # (iii) sample sharding: two half-size sample ranges (offset i0) summed by the finalize
    #       kernel's multi-buffer path agree with the single-range result to fp32 summation noise
    half = N // 2
    wsA = smoothing.Workspace(s, smoothing.ZERO_ORDER, T, half)
    both = _device.empty((2,) + tuple(wsA.partials.shape), torch.float32)
    for r in range(2):
        smoothing.accumulate(s, smoothing.ZERO_ORDER, x_nom, u_nom, half, wsA, i0=r * half, **kw)
        both[r].copy_(wsA.partials)
    A3, B3, c3, st3 = smoothing.finalize(s, smoothing.ZERO_ORDER, x_nom, u_nom, wsA, N, partials=both,
                                         nranks=2, rank_stride=wsA.partials.numel())
    assert int(st3.sum().item()) == 0
    assert rel_err(_device.to_numpy(A3), _device.to_numpy(A1)) < 1e-5
    assert rel_err(_device.to_numpy(B3), _device.to_numpy(B1)) < 1e-5
    # (iv) smoothing converges to the exact Jacobian as sigma -> 0 (quadrotor is smooth)
    if name == "quadrotor":
        A4, B4, c4, _ = run(x_nom, u_nom, N, sigma=1e-2 * np.ones(16))
        Ae, Be, ce = solver.get_TV_matrices(x_trj, cfg["u_trj_initial"])
        assert rel_err(_device.to_numpy(A4), Ae) < 2e-3
        assert rel_err(_device.to_numpy(B4), Be) < 2e-3


@pytest.mark.parametrize("zero_sigma", [True, False])
@pytest.mark.parametrize("name,N", [("pendulum", 700), ("bicycle", 700), ("three_cart", 5000), ("quadrotor", 5000)])
def test_finalize_variants_are_bit_identical(api, name, N, zero_sigma, monkeypatch):
    """The two finalize kernels (one block per point for few points, four threads per point for many)
    perform the same fp64 operations in the same order: a point's (A, B, c) must not depend on how
    many points a launch holds (instance / timestep sharding relies on it).  With zero_sigma one
    regressor is given sigma = 0 to take the zero-column branch (which also makes every update with
    that column exact — the all-nonzero case is the one that catches a multiply-add the compiler did
    not contract); the point count is ragged against the 32-point blocks, and N spans two chunks for
    the larger systems."""
    import torch
    from irs_mpc_b200 import _device, smoothing
    P = 1300                                   # > 8 * 148: the launch would pick the quad variant
    cfg = ec.CONFIGS[name](T=4)
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    rng = np.random.default_rng(77)
    x_nom = _device.to_device(cfg["x0"] + 0.1 * rng.standard_normal((P, n)))
    u_nom = _device.to_device(cfg["u_trj_initial"][0] + 0.1 * rng.standard_normal((P, m)))
    sigma = np.array(cfg["sigma"], dtype=np.float64).copy()
    if zero_sigma:
        sigma[1] = 0.0
    ws = smoothing.Workspace(s, smoothing.ZERO_ORDER, P, N)
    smoothing.accumulate(s, smoothing.ZERO_ORDER, x_nom, u_nom, N, ws, sigma=sigma, seed=5, it=1)
    out = {}
    for variant in ("block", "quad"):
        monkeypatch.setenv("IRS_FINALIZE_VARIANT", variant)
        At, Bt, ct, status = smoothing.finalize(s, smoothing.ZERO_ORDER, x_nom, u_nom, ws, N)
        assert int(status.sum().item()) == 0
        out[variant] = (At.clone(), Bt.clone(), ct.clone())
    for a, b in zip(out["block"], out["quad"]):
        assert torch.equal(a, b)
    assert float(out["quad"][0].abs().max()) > 0 and bool(torch.isfinite(out["quad"][0]).all())
    if zero_sigma:
        assert float(out["quad"][0][:, :, 1].abs().max()) == 0.0    # zero regressor -> zero coefficient
    monkeypatch.delenv("IRS_FINALIZE_VARIANT")
    few = 100                                  # few points: the launch picks the block variant itself
    At, Bt, ct, status = smoothing.finalize(s, smoothing.ZERO_ORDER, x_nom[:few].contiguous(),
                                            u_nom[:few].contiguous(), ws, N, partials=ws.partials[:few])
    for a, b in zip((At, Bt, ct), out["quad"]):
        assert torch.equal(a[:few], b[:few])
    # the multi-rank inputs of the sample-sharded path: two fp32 partial buffers (summed in rank
    # order), and two fp64 chunk-reduced blocks (what the ranks exchange)
    both = _device.empty((2,) + tuple(ws.partials.shape), torch.float32)
    red = _device.empty((2, P, ws.width))
    both[0].copy_(ws.partials)
    smoothing.reduce_chunks(s, smoothing.ZERO_ORDER, ws, out=red[0])
    smoothing.accumulate(s, smoothing.ZERO_ORDER, x_nom, u_nom, N, ws, sigma=sigma, seed=5, it=1, i0=N)
    both[1].copy_(ws.partials)
    smoothing.reduce_chunks(s, smoothing.ZERO_ORDER, ws, out=red[1])
    for kw in (dict(partials=both, nranks=2, rank_stride=ws.partials.numel()),
               dict(reduced=red, nranks=2, rank_stride=red[0].numel())):
        res = {}
        for variant in ("block", "quad"):
            monkeypatch.setenv("IRS_FINALIZE_VARIANT", variant)
            At, Bt, ct, status = smoothing.finalize(s, smoothing.ZERO_ORDER, x_nom, u_nom, ws, 2 * N, **kw)
            assert int(status.sum().item()) == 0
            res[variant] = (At.clone(), Bt.clone(), ct.clone())
        for a, b in zip(res["block"], res["quad"]):
            assert torch.equal(a, b)
        assert bool(torch.isfinite(res["quad"][0]).all()) and float(res["quad"][0].abs().max()) > 0
    ws.partials.copy_(both[0])
    # a point whose Gram block is not finite is flagged (status 1) by both variants, and only that point
    ws.partials[7].fill_(float("nan"))
    for variant in ("block", "quad"):
        monkeypatch.setenv("IRS_FINALIZE_VARIANT", variant)
        status = smoothing.finalize(s, smoothing.ZERO_ORDER, x_nom, u_nom, ws, N)[3]
        st = _device.to_numpy(status)
        assert st[7] == 1 and st.sum() == 1


# ------------------------------------------------------------------------------------------------
# batched MPC instances (BASELINE.json configs[4])
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,I,T,N", [("quadrotor", 5, 24, 8192), ("pendulum", 300, 30, 600)])
def test_batched_instances_match_oracle_and_shard(api, name, I, T, N):
    """Every instance of a batch equals the single-problem oracle pipeline on the deltas the kernel
    drew for it (1e-4), and a shard of the batch (instance_offset) is bit-identical to the same
    instances inside the full batch — what instance sharding over GPUs relies on."""
    import torch
    from irs_mpc_b200 import _device
    cfg = ec.CONFIGS[name](T=T)
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    rng = np.random.default_rng(5000)
    x0 = cfg["x0"] + 0.02 * rng.standard_normal((I, n))
    shift = np.zeros(n)
    shift[0] = 1.0
    xd = np.stack([cfg["xd_trj"] + (0.2 * b / I) * shift for b in range(I)])   # per-instance targets
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=77)
    batch = api.BatchedIrsLqrZeroOrder(s, cfg["Q"], cfg["Qd"], cfg["R"], x0, xd, cfg["u_trj_initial"], sampler)
    x_init = _device.to_numpy(batch.x_trj)
    x_new, u_new, cost_new = batch.local_descent()
    batch.check()
    x_new, u_new, cost_new = _device.to_numpy(x_new), _device.to_numpy(u_new), _device.to_numpy(cost_new)
    orc = cr.SYSTEMS[name](s.h)
    for b in sorted(set([0, 1, I // 2, I - 1])):
        np.testing.assert_allclose(x_init[b], cr.rollout(orc, x0[b], cfg["u_trj_initial"]), rtol=1e-12, atol=1e-12)
        deltas = sampler.deltas(T, 1, t0=b * T).astype(np.float64)
        At, Bt, ct = cr.zero_order_tv_matrices(orc, x_init[b], cfg["u_trj_initial"], deltas)
        K, k = cr.tvlqr_riccati(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], xd[b])
        x_o, u_o = cr.closed_loop_descent(orc, K, k, x_init[b][0])
        cost_o = cr.evaluate_cost(x_o, u_o, xd[b], cfg["Q"], cfg["R"])
        assert rel_err(x_new[b], x_o) < FP32_RTOL
        assert rel_err(u_new[b], u_o) < 5 * FP32_RTOL
        assert abs(cost_new[b] - cost_o) / abs(cost_o) < FP32_RTOL
    # shard [lo, hi) with instance_offset = lo
    lo, hi = 1, min(I, 4)
    shard = api.BatchedIrsLqrZeroOrder(s, cfg["Q"], cfg["Qd"], cfg["R"], x0[lo:hi], xd[lo:hi],
                                       cfg["u_trj_initial"], sampler, instance_offset=lo)
    xs, us, cs = shard.local_descent()
    shard.check()
    assert np.array_equal(_device.to_numpy(xs), x_new[lo:hi])
    assert np.array_equal(_device.to_numpy(us), u_new[lo:hi])
    assert np.array_equal(_device.to_numpy(cs), cost_new[lo:hi])
    # iterate() keeps the reference's bookkeeping: k + 1 descents, k + 2 cost entries
    xk, uk, ck = batch.iterate(1)
    assert len(batch.cost_lst) == 3 and xk.shape == (I, T + 1, n) and ck.shape == (I,)
    assert np.all(np.isfinite(ck))


# ------------------------------------------------------------------------------------------------
# CUDA-graph replay of the per-iteration call sequence
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,T,N", [("pendulum", 60, 1000), ("quadrotor", 30, 2000)])
def test_graph_replay_is_bit_identical_to_eager(api, name, T, N):
    """From the third call on, local_descent / get_TV_matrices are replayed from a CUDA graph whose
    accumulate node is re-parameterised (iter, seed, sigma) — the results must equal the eager
    launches bit for bit, iteration after iteration."""
    from irs_mpc_b200 import _graph as mod
    cfg = ec.CONFIGS[name](T=T)
    n = cfg["x0"].shape[0]

    def run(use_graphs):
        old = mod.USE_GRAPHS
        mod.USE_GRAPHS = use_graphs
        try:
            s = make_system(api, name)
            sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=11)
            solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=T), sampler)
            solver.iterate(5, verbose=False)
            tv = []
            for k in range(4):
                sampler.seed = 100 + k
                tv.append(solver.get_TV_matrices(solver.x_trj, solver.u_trj))
            return solver, tv
        finally:
            mod.USE_GRAPHS = old

    eager, tv_e = run(False)
    graph, tv_g = run(True)
    slots = graph._graphs._slots
    assert "descent" in slots and slots["descent"][1] is not None      # really replayed
    assert "linearize" in slots and slots["linearize"][1] is not None
    assert not eager._graphs._slots
    assert eager.cost_lst == graph.cost_lst
    for a, b in zip(eager.x_trj_lst, graph.x_trj_lst):
        assert np.array_equal(a, b)
    for (A1, B1, c1), (A2, B2, c2) in zip(tv_e, tv_g):
        assert np.array_equal(A1, A2) and np.array_equal(B1, B2) and np.array_equal(c1, c2)


@pytest.mark.parametrize("I", [1, 37])
def test_quadrotor_rollout_with_trig_ahead_is_bit_identical(api, I, monkeypatch):
    """The quadrotor rollouts evaluate sin / cos of the next Euler angles one step ahead on a second
    warp (rollout_trig_kernel); trajectories, inputs and costs must equal the one-warp kernel's."""
    import torch
    from irs_mpc_b200 import _device, _lib
    cfg = ec.CONFIGS["quadrotor"](T=60)
    s = make_system(api, "quadrotor")
    n, m, T = 12, 4, 60
    rng = np.random.default_rng(9)
    K = _device.to_device(1e-3 * rng.standard_normal((I, T, m, n)))      # weak feedback: the flight stays tame
    k = _device.to_device(cfg["u_trj_initial"][None, :T] + 0.02 * rng.standard_normal((I, T, m)))
    x0 = _device.to_device(cfg["x0"] + 0.05 * rng.standard_normal((I, n)))
    xd = _device.to_device(cfg["xd_trj"][:T + 1])
    Q, R = _device.to_device(cfg["Q"]), _device.to_device(cfg["R"])
    prm, nprm = s._params()
    out = {}
    for flag in ("0", "1"):
        monkeypatch.setenv("IRS_ROLLOUT_TRIG", flag)
        xs, us, cost = _device.empty((I, T + 1, n)), _device.empty((I, T, m)), _device.empty((I,))
        _lib.call("irs_rollout_closed_loop", s.system_id, prm, nprm, _device.ptr(K), _device.ptr(k), _device.ptr(x0),
                  _device.ptr(xd), 0, _device.ptr(Q), _device.ptr(R), I, T, _device.ptr(xs), _device.ptr(us),
                  _device.ptr(cost), _device.stream_ptr())
        xo, co = _device.empty((I, T + 1, n)), _device.empty((I,))
        _lib.call("irs_rollout_open_loop", s.system_id, prm, nprm, _device.ptr(us), _device.ptr(x0),
                  _device.ptr(xd), 0, _device.ptr(Q), _device.ptr(R), I, T, _device.ptr(xo), _device.ptr(co),
                  _device.stream_ptr())
        out[flag] = (xs, us, cost, xo, co)
    assert all(bool(torch.isfinite(v).all()) for v in out["0"])
    for a, b in zip(out["0"], out["1"]):
        assert torch.equal(a, b)
    assert torch.equal(out["1"][0], out["1"][3])      # the open-loop rollout of the applied inputs replays the closed loop
    assert float((out["1"][0][:, -1, 3:6]).abs().max()) > 1e-3            # the attitude really moved


@pytest.mark.parametrize("n,m", [(12, 4), (6, 2)])
def test_riccati_segments_chain_to_the_full_pass(api, n, m):
    """irs_tvlqr_riccati_segment over [t1,T), [t2,t1), [0,t2) with the carried (P, p) reproduces the
    one-launch backward pass bit for bit (what the pipelined descent relies on)."""
    import torch
    from irs_mpc_b200 import _device, _lib, tv_lqr
    I, T = 3, 37
    rng = np.random.default_rng(3)
    At = _device.to_device(np.eye(n) + 0.05 * rng.standard_normal((I, T, n, n)))
    Bt = _device.to_device(0.1 * rng.standard_normal((I, T, n, m)))
    ct = _device.to_device(0.01 * rng.standard_normal((I, T, n)))
    Q, Qd, R = (_device.to_device(v) for v in (np.eye(n), 10 * np.eye(n), 0.1 * np.eye(m)))
    xd = _device.to_device(rng.standard_normal((I, T + 1, n)))
    K0, k0, st0 = tv_lqr.riccati_device(At, Bt, ct, Q, Qd, R, xd, (T + 1) * n)
    K = torch.full_like(K0, float("nan"))
    k = torch.full_like(k0, float("nan"))
    st = _device.empty((I,), torch.int32)
    carry = _device.empty((I, n * n + n))
    for lo, hi in ((25, 37), (11, 25), (0, 11)):
        _lib.call("irs_tvlqr_riccati_segment", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                  _device.ptr(Q), _device.ptr(Qd), _device.ptr(R), _device.ptr(xd), (T + 1) * n, I, T, lo, hi,
                  _device.ptr(carry), _device.ptr(K), _device.ptr(k), _device.ptr(st), _device.stream_ptr())
    assert torch.equal(K, K0) and torch.equal(k, k0) and int(st.sum().item()) == 0 == int(st0.sum().item())
    # a partial segment without the carry buffer is refused
    with pytest.raises(_lib.IrsCudaError, match="carry"):
        _lib.call("irs_tvlqr_riccati_segment", n, m, _device.ptr(At), _device.ptr(Bt), _device.ptr(ct),
                  _device.ptr(Q), _device.ptr(Qd), _device.ptr(R), _device.ptr(xd), (T + 1) * n, I, T, 5, T,
                  None, _device.ptr(K), _device.ptr(k), _device.ptr(st), _device.stream_ptr())


@pytest.mark.parametrize("name,T,N,graphs,order", [("quadrotor", 30, 2000, True, 0), ("quadrotor", 30, 2000, False, 0),
                                                   ("three_cart", 40, 3000, True, 0), ("quadrotor", 30, 500, True, 1)])
def test_pipelined_descent_is_bit_identical_to_one_pass(api, name, T, N, graphs, order):
    """local_descent linearizes the horizon in three launches from the back and runs each segment's
    fit + Riccati steps on a second stream (irs_lqr._SampledIrsLqr._pipeline_segments); the iterates
    must equal those of the one-pass sequence bit for bit, eagerly and replayed from a CUDA graph."""
    from irs_mpc_b200 import _graph as gmod
    from irs_mpc_b200 import irs_lqr as mod
    cfg = ec.CONFIGS[name](T=T)
    n = cfg["x0"].shape[0]

    def run(pipeline):
        old = mod._USE_PIPELINE, gmod.USE_GRAPHS, mod._PIPELINE_SEGMENTS
        mod._USE_PIPELINE, gmod.USE_GRAPHS, mod._PIPELINE_SEGMENTS = pipeline, graphs, 3    # forced: the test problem is small
        try:
            s = make_system(api, name)
            sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=23,
                                           projection="delta" if name == "three_cart" else None)
            cls = api.IrsLqrZeroOrder if order == 0 else api.IrsLqrFirstOrder
            solver = cls(s, make_params(api, cfg, T=T), sampler)
            assert (solver._pipeline_segments() is not None) == pipeline
            solver.iterate(4, verbose=False)
            return solver
        finally:
            mod._USE_PIPELINE, gmod.USE_GRAPHS, mod._PIPELINE_SEGMENTS = old

    one, pipe = run(False), run(True)
    assert one.cost_lst == pipe.cost_lst
    for a, b in zip(one.x_trj_lst, pipe.x_trj_lst):
        assert np.array_equal(a, b)
    for a, b in zip(one.u_trj_lst, pipe.u_trj_lst):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------------------------------------
# CEM baseline (irs_lqr/cem.py) — SURVEY.md section 8f row 2
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,T,B", [("pendulum", 60, 200), ("three_cart", 40, 128), ("bicycle", 40, 300),
                                      ("quadrotor", 30, 1000)])
def test_cem_matches_numpy_restatement(api, name, T, B):
    """Same seed -> same candidates (np.random.normal, as the reference); costs from the batched
    rollout kernel equal the float64 loop of cem.py:165-169, so the elite set and the refit agree."""
    from irs_mpc_b200 import _device
    cfg = ec.CONFIGS[name](T=T)
    s = make_system(api, name)
    m = s.dim_u
    p = api.CemParameters()
    p.Q, p.Qd, p.R, p.x0, p.xd_trj, p.u_trj_initial = (cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"],
                                                       cfg["u_trj_initial"])
    p.n_elite, p.batch_size, p.initial_std = 20, B, 0.5 * np.ones(m)
    np.random.seed(1234)
    solver = api.CrossEntropyMethod(s, p)
    x_new, u_new = solver.local_descent(solver.x_trj, solver.u_trj)
    # restatement of cem.py:151-184 on the oracle dynamics
    orc = cr.SYSTEMS[name](s.h)
    np.random.seed(1234)
    cand = np.random.normal(cfg["u_trj_initial"], np.tile(p.initial_std, (T, 1)), (B, T, m))
    costs = np.array([cr.evaluate_cost(cr.rollout(orc, cfg["x0"], cand[k]), cand[k], cfg["xd_trj"], cfg["Q"],
                                       cfg["R"]) for k in range(B)])
    best = np.argpartition(costs, p.n_elite)[:p.n_elite]
    # the device's elites are the first n_elite of the stable order (NaN last, ties by index)
    want = np.zeros(B, np.int32)
    want[np.argsort(costs, kind="stable")[:p.n_elite]] = 1
    assert np.array_equal(_device.to_numpy(solver.last_elite), want)
    u_o = cand[best].mean(axis=0)
    np.testing.assert_allclose(u_new, u_o, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(solver.std_trj, cand[best].std(axis=0), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(x_new, cr.rollout(orc, cfg["x0"], u_o), rtol=1e-9, atol=1e-9)
    x, u, c = solver.iterate(2, verbose=False)
    assert len(solver.cost_lst) == 4 and np.isfinite(c)


@pytest.mark.parametrize("name", SYSTEMS)
def test_compute_least_squares_matches_lstsq(api, name):
    """IrsLqrZeroOrder.compute_least_squares (irs_lqr_zero_order.py:27-36) on explicit samples: the
    library's fp64 Gram block + Cholesky fit against np.linalg.lstsq (the reference's call)."""
    cfg = ec.CONFIGS[name](T=6)
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], 500, seed=1)
    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=6), sampler)
    rng = np.random.default_rng(8)
    dxdu = rng.standard_normal((700, n + m)) * cfg["sigma"]
    AB_true = rng.standard_normal((n, n + m))
    deltaf = dxdu @ AB_true.T + 1e-3 * rng.standard_normal((700, n))
    A, B = solver.compute_least_squares(dxdu, deltaf)
    AB = np.linalg.lstsq(dxdu, deltaf, rcond=None)[0].T
    assert A.shape == (n, n) and B.shape == (n, m)
    np.testing.assert_allclose(np.hstack((A, B)), AB, rtol=0, atol=1e-9 * max(1.0, float(np.max(np.abs(AB)))))
    with pytest.raises(np.linalg.LinAlgError):
        solver.compute_least_squares(dxdu[:n + m - 1], deltaf[:n + m - 1])      # fewer samples than regressors


def test_batched_instances_bounds_are_checked(api):
    """BatchedIrsLqrZeroOrder with the reference's xbound / ubound: wide boxes (the examples' 'infinite'
    1e5) change nothing; a box that a planned trajectory touches is reported by check() as the reference's
    ValueError, naming the instances — never a silently unconstrained result."""
    from irs_mpc_b200 import _device
    I, T, N = 6, 20, 2000
    cfg = ec.quadrotor(T=T)
    s = make_system(api, "quadrotor")
    x0, xd = ec.quadrotor_batch(0, I, T=T, total=64)
    mk = lambda **kw: api.BatchedIrsLqrZeroOrder(
        s, cfg["Q"], cfg["Qd"], cfg["R"], x0, xd, cfg["u_trj_initial"],
        api.GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], N, seed=3), **kw)
    free = mk()
    xf, uf, cf = free.local_descent()
    free.check()
    wide = mk(xbound=cfg["xbound"], ubound=cfg["ubound"])
    xw, uw, cw = wide.local_descent()
    wide.check()
    assert np.array_equal(_device.to_numpy(xf), _device.to_numpy(xw)) and np.array_equal(_device.to_numpy(cf), _device.to_numpy(cw))
    umax = float(np.max(np.abs(_device.to_numpy(uf))))
    tight = mk(xbound=cfg["xbound"], ubound=np.array([-0.5 * umax * np.ones(4), 0.5 * umax * np.ones(4)]))
    tight.local_descent()
    with pytest.raises(ValueError, match="TV_LQR failed"):
        tight.check()


def test_integration_stub_runs_as_documented(api, golden_dir):
    """INTEGRATION.md section B shows the binding a reference maintainer would add (ctypes against the C
    ABI, nothing from this package).  The code block is read out of the document and executed as written;
    its (At, Bt, ct) on the reference-generated deltas must equal the reference's own."""
    import re
    from irs_mpc_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    block = re.search(r"```python\n# irs_lqr/_b200.py.*?\n(.*?)```", text, flags=re.S).group(1)
    block = block.replace('ctypes.CDLL("libirs_mpc_b200.so")', 'ctypes.CDLL(%r)' % _lib.LIB_PATH)
    ns = {}
    exec(compile(block, "INTEGRATION.md:_b200.py", "exec"), ns)
    g = gold(golden_dir, "zero_order_quadrotor.npz")
    params = [0.05, 0.775, 0.15, 9.81, 0.0015, 0.0025, 0.0035, 1.0, 0.0245]
    At, Bt, ct = ns["zero_order_tv_matrices"](2, params, g["x_trj"], g["u_trj"], g["deltas"])
    assert rel_err(At, g["At"]) < FP32_RTOL and rel_err(Bt, g["Bt"]) < FP32_RTOL
    assert float(np.max(np.abs(ct - g["ct"]))) < FP32_RTOL * max(1.0, float(np.max(np.abs(g["x_trj"]))))


# ------------------------------------------------------------------------------------------------
# ragged / edge sample counts through both Gram engines
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("name,N", [("quadrotor", 17), ("quadrotor", 127), ("quadrotor", 128), ("quadrotor", 129),
                                    ("quadrotor", 255), ("quadrotor", 256), ("quadrotor", 257),
                                    ("quadrotor", 4097), ("quadrotor", 8191), ("quadrotor", 35), ("pendulum", 4),
                                    ("pendulum", 9), ("pendulum", 33), ("bicycle", 300), ("three_cart", 257)])
def test_ragged_sample_counts_match_oracle(api, name, N, engine, antithetic):
    """Sample counts that do not fill a 32-sample warp tile, a 128-sample block round (256 samples when a
    lane owns an antithetic pair) or a 4096-sample chunk: the padded lanes must contribute nothing, and
    an odd count ends in a lone + member (fit vs the fp64 oracle on the same deltas)."""
    from irs_mpc_b200 import _device, _lib, smoothing
    T = 3
    cfg, s, u_trj = _nominal(api, name, T)
    n = s.dim_x
    if antithetic and N < 2 * (n + s.dim_u) + 2:
        pytest.skip("N antithetic samples span only ceil(N/2) directions: the fit needs N >= 2 (n + m)")
    x_trj = cr.rollout(cr.SYSTEMS[name](s.h), cfg["x0"], u_trj)
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=5,
                                   antithetic=antithetic)
    _lib.call("irs_set_gram_engine", engine)
    try:
        At, Bt, ct, status, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, _device.to_device(x_trj[:T]),
                                                    _device.to_device(u_trj), N, sigma=sampler.sigma(1),
                                                    seed=sampler.seed, it=1, flags=sampler.flags())
        assert int(status.sum().item()) == 0
        At, Bt, ct = _device.to_numpy(At), _device.to_numpy(Bt), _device.to_numpy(ct)
    finally:
        _lib.call("irs_set_gram_engine", -1)
    deltas = sampler.deltas(T, 1).astype(np.float64)
    Ao, Bo, co = cr.zero_order_tv_matrices(cr.SYSTEMS[name](s.h), x_trj, u_trj, deltas)
    # few samples -> ill-conditioned normal equations amplify the fp32 Gram noise
    tol = FP32_RTOL * (30.0 if N < 3 * (n + s.dim_u) else 1.0)
    assert rel_err(At, Ao) < tol
    assert rel_err(Bt, Bo) < tol
    assert float(np.max(np.abs(ct - co))) < tol * max(1.0, float(np.max(np.abs(x_trj))))


@pytest.mark.parametrize("engine", [0, 1])
@pytest.mark.parametrize("name,projection,N", [("quadrotor", None, 9001), ("quadrotor", None, 12288),
                                               ("three_cart", None, 5001), ("three_cart", "absolute", 5001),
                                               ("three_cart", "delta", 8192), ("pendulum", None, 777),
                                               ("bicycle", None, 1001)])
def test_antithetic_pairs_equal_the_replay_of_their_own_deltas(api, name, projection, N, engine):
    """The paired kernel (one Philox draw and — without projection — ONE operand row per pair, regressor
    block doubled at read-back, lone + member scaled by sqrt 2) against the ordinary one-row-per-sample
    kernel fed, through the replay path, with the deltas of the same antithetic stream: both are fp32
    accumulations of the same sums, so they agree far inside the 1e-4 budget; the index bookkeeping of
    the pairs (which counter, which sign, which samples exist) would show up as O(1) differences."""
    import torch
    from irs_mpc_b200 import _device, _lib, smoothing
    T = 3
    cfg, s, u_trj = _nominal(api, name, T)
    n = s.dim_x
    x_trj = cr.rollout(cr.SYSTEMS[name](s.h), cfg["x0"], u_trj)
    x_nom, u_nom = _device.to_device(x_trj[:T]), _device.to_device(u_trj)
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=31,
                                   projection=projection, antithetic=True)
    noise = _device.to_device(sampler.deltas(T, 2), torch.float32)
    proj_flags = sampler.flags() & 6
    _lib.call("irs_set_gram_engine", engine)
    try:
        Ap, Bp, cp, st, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x_nom, u_nom, N, sigma=sampler.sigma(2),
                                                seed=sampler.seed, it=2, flags=sampler.flags())
        assert int(st.sum().item()) == 0
        Ap, Bp, cp = _device.to_numpy(Ap), _device.to_numpy(Bp), _device.to_numpy(cp)
        Ar, Br, cr_, st, _ = smoothing.linearize(s, smoothing.ZERO_ORDER, x_nom, u_nom, N, noise=noise,
                                                 flags=proj_flags)
        assert int(st.sum().item()) == 0
        Ar, Br, cr_ = _device.to_numpy(Ar), _device.to_numpy(Br), _device.to_numpy(cr_)
    finally:
        _lib.call("irs_set_gram_engine", -1)
    # bicycle on the tensor-core engine (not its default): its steer regressor has sigma 0.01 next to
    # sigma 2 columns, and the 2^-17 product noise of the bf16x2 split on the cross terms is then ~1e-4 of
    # that column's own Gram entry — both kernels carry it, independently
    tol = 3e-4 if (name == "bicycle" and engine == 1) else 2e-5
    assert rel_err(Ap, Ar) < tol and rel_err(Bp, Br) < tol
    assert float(np.max(np.abs(cp - cr_))) < tol * max(1.0, float(np.max(np.abs(x_trj))))


# ------------------------------------------------------------------------------------------------
# box-constrained TVLQR (SURVEY.md section 8f row 1): irs_lqr/tv_lqr.py:113-118,:132-134
# ------------------------------------------------------------------------------------------------
def _bicycle_lin(T, u_const):
    cfg = ec.bicycle(T=T)
    orc = cr.BicycleOracle(cfg["h"])
    u0 = np.tile(np.array(u_const), (T, 1))
    x_trj = cr.rollout(orc, cfg["x0"], u0)
    At, Bt, ct = cr.exact_tv_matrices(orc, x_trj, u0)
    return cfg, orc, At, Bt, ct


def test_solve_tvlqr_active_bounds_matches_admm_oracle_and_dense_qp(api):
    """One QP with an active steer / steer-rate box: the CUDA ADMM against the numpy ADMM (1e-7) and
    against an independent dense QP solve (scipy SLSQP, 1e-5); the plan obeys the bounds."""
    from oracle import box_tvlqr as bq
    T = 12
    cfg, orc, At, Bt, ct = _bicycle_lin(T, [0.5, 0.6])
    xlo, xhi = np.array([-1e4, -1e4, -1e4, -1e4, -0.3]), np.array([1e4, 1e4, 1e4, 1e4, 0.3])
    ulo, uhi = np.array([-1e4, -0.4]), np.array([1e4, 0.4])
    xb = np.stack((np.tile(xlo, (T + 1, 1)), np.tile(xhi, (T + 1, 1))))
    ub = np.stack((np.tile(ulo, (T, 1)), np.tile(uhi, (T, 1))))
    xs, us = api.solve_tvlqr(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], None,
                             x_bound_abs=xb, u_bound_abs=ub)
    xo, uo, _ = bq.admm_box_qp(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], xlo, xhi, ulo, uhi)
    np.testing.assert_allclose(xs, xo, rtol=0, atol=1e-7)
    np.testing.assert_allclose(us, uo, rtol=0, atol=1e-7)
    xr, ur, res = bq.dense_qp_reference(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], xlo, xhi,
                                        ulo, uhi)
    assert res.success
    np.testing.assert_allclose(us, ur, rtol=0, atol=2e-5)
    np.testing.assert_allclose(xs, xr, rtol=0, atol=2e-5)
    assert np.all(xs[1:, 4] <= 0.3 + 1e-6) and np.all(np.abs(us[:, 1]) <= 0.4 + 1e-6)
    assert np.max(np.abs(xs[:, 4])) > 0.29          # the bound really is active
    # inactive bounds still take the exact one-pass path and agree with the unbounded call
    wide = np.stack((np.tile(-1e4 * np.ones(5), (T + 1, 1)), np.tile(1e4 * np.ones(5), (T + 1, 1))))
    x1, u1 = api.solve_tvlqr(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], None,
                             x_bound_abs=wide)
    x2, u2 = api.solve_tvlqr(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], None)
    assert np.array_equal(x1, x2) and np.array_equal(u1, u2)


def test_solve_tvlqr_time_varying_and_relative_bounds(api):
    """tv_lqr.py:113-124: the reference indexes its boxes by timestep.  A steer box that tightens over
    the horizon and a steer-rate box that opens up, against the numpy ADMM and the dense QP solve; the
    start-state box (an x0 outside it is an infeasible QP) and the relative bounds (free variables when
    indices_u_into_x is None: inert unless empty)."""
    from oracle import box_tvlqr as bq
    T = 12
    cfg, orc, At, Bt, ct = _bicycle_lin(T, [0.5, 0.6])
    steer = np.linspace(0.45, 0.2, T + 1)
    rate = np.linspace(0.25, 0.6, T)
    xhi = np.tile(np.array([1e4, 1e4, 1e4, 1e4, 0.0]), (T + 1, 1))
    xhi[:, 4] = steer
    xlo = -xhi
    uhi = np.tile(np.array([1e4, 0.0]), (T, 1))
    uhi[:, 1] = rate
    ulo = -uhi
    args = (At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"])
    xs, us = api.solve_tvlqr(*args, None, x_bound_abs=np.stack((xlo, xhi)), u_bound_abs=np.stack((ulo, uhi)))
    xo, uo, _ = bq.admm_box_qp(*args, xlo, xhi, ulo, uhi)
    np.testing.assert_allclose(xs, xo, rtol=0, atol=1e-7)
    np.testing.assert_allclose(us, uo, rtol=0, atol=1e-7)
    xr, ur, res = bq.dense_qp_reference(*args, xlo, xhi, ulo, uhi)
    assert res.success
    np.testing.assert_allclose(us, ur, rtol=0, atol=2e-5)
    np.testing.assert_allclose(xs, xr, rtol=0, atol=2e-5)
    assert np.all(np.abs(xs[1:, 4]) <= steer[1:] + 1e-6) and np.all(np.abs(us[:, 1]) <= rate + 1e-6)
    assert np.sum(np.abs(xs[1:, 4]) > steer[1:] - 1e-4) >= 2      # active at more than one timestep
    # relative bounds with indices_u_into_x=None bound free variables: no effect ...
    rel_x = np.stack((-1e-3 * np.ones((T, 5)), 1e-3 * np.ones((T, 5))))
    rel_u = np.stack((-1e-3 * np.ones((T, 2)), 1e-3 * np.ones((T, 2))))
    x1, u1 = api.solve_tvlqr(*args, None, x_bound_rel=rel_x, u_bound_rel=rel_u)
    x2, u2 = api.solve_tvlqr(*args, None)
    assert np.array_equal(x1, x2) and np.array_equal(u1, u2)
    # ... unless they are empty (infeasible program)
    with pytest.raises(ValueError, match="TV_LQR failed"):
        api.solve_tvlqr(*args, None, x_bound_rel=np.stack((1e-3 * np.ones((T, 5)), -1e-3 * np.ones((T, 5)))))
    # x_0 is boxed as well (tv_lqr.py:113-114 at t = 0)
    tight = np.stack((np.tile(cfg["x0"] + 0.5, (T + 1, 1)), np.tile(cfg["x0"] + 1e4, (T + 1, 1))))
    with pytest.raises(ValueError, match="TV_LQR failed"):
        api.solve_tvlqr(*args, None, x_bound_abs=tight)
    with pytest.raises(NotImplementedError):
        api.solve_tvlqr(*args, None, indices_u_into_x=np.array([0, 1]))


def test_bicycle_descent_with_active_steer_bound_matches_oracle(api):
    """The bicycle example's +-pi/4 steer bound (bicycle_first_order.py:23-26) is active: local_descent
    must run the reference's loop (box QP at every timestep, first input on the true dynamics).
    Checked against the numpy restatement of that loop; the result obeys the bound and lowers the cost."""
    from oracle import box_tvlqr as bq
    T = 40
    cfg = ec.bicycle(T=T)
    s = make_system(api, "bicycle")
    solver = api.IrsLqrExact(s, make_params(api, cfg, T=T))
    x_new, u_new = solver.local_descent(solver.x_trj, solver.u_trj)
    cost = solver.evaluate_cost(x_new, u_new)
    assert solver.bounded_admm_iterations > 0              # the bounded path ran
    orc = cr.BicycleOracle(cfg["h"])
    At, Bt, ct = cr.exact_tv_matrices(orc, solver.x_trj, solver.u_trj)
    gains0 = cr.tvlqr_riccati(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["xd_trj"])
    xo, uo, _ = bq.mpc_box_descent(orc, At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"],
                                   cfg["xbound"][0], cfg["xbound"][1], cfg["ubound"][0], cfg["ubound"][1],
                                   gains0=gains0)
    np.testing.assert_allclose(u_new, uo, rtol=0, atol=1e-6)
    np.testing.assert_allclose(x_new, xo, rtol=0, atol=1e-6)
    assert np.max(np.abs(x_new[:, 4])) <= np.pi / 4 + 1e-6
    assert np.max(np.abs(x_new[:, 4])) > np.pi / 4 - 1e-3
    assert cost < solver.cost
    # the whole bicycle loop now runs end to end (it raised NotImplementedError before)
    solver.iterate(3, verbose=False)
    assert len(solver.cost_lst) == 5 and np.all(np.isfinite(solver.cost_lst))
    assert solver.cost_lst[-1] < solver.cost_lst[0]


def test_plan_check_keeps_unbounded_problems_on_the_exact_path(api):
    """Quadrotor / pendulum examples pass 'infinite' boxes (1e4, 1e5): no plan touches them, the
    one-pass Riccati descent is used and equals the run without any bounds bit for bit."""
    cfg = ec.pendulum(T=60)
    s = make_system(api, "pendulum")
    a = api.IrsLqrExact(s, make_params(api, cfg, T=60))
    p2 = make_params(api, cfg, T=60)
    p2.xbound, p2.ubound = None, None
    b = api.IrsLqrExact(s, p2)
    xa, ua = a.local_descent(a.x_trj, a.u_trj)
    xb_, ub_ = b.local_descent(b.x_trj, b.u_trj)
    assert np.array_equal(xa, xb_) and np.array_equal(ua, ub_)
    assert not hasattr(a, "bounded_admm_iterations")


def test_bicycle_exact_loop_lands_on_the_stored_curve(api, golden_dir):
    """examples/bicycle/analysis/bicycle_easy_exact.csv: entry 0 is reproduced exactly; the later
    entries depend on OSQP's 1e-3 tolerance (parity unpinned, SURVEY.md section 4: an accurate box QP
    lands 0.7 % - 10 % away), so only the converged level is compared (3 %)."""
    goldc = np.array(json.load(open(os.path.join(golden_dir, "reference_costs.json")))
                     ["stored_cost_curves"]["bicycle_easy_exact"]["values"])
    cfg = ec.bicycle(T=100)
    solver = api.IrsLqrExact(make_system(api, "bicycle"), make_params(api, cfg, T=100))
    assert abs(solver.cost - goldc[0]) <= 1e-9 * goldc[0]
    solver.iterate(len(goldc) - 2, verbose=False)
    assert len(solver.cost_lst) == len(goldc)
    assert abs(solver.cost_lst[-1] - goldc[-1]) <= 0.03 * goldc[-1]
    assert np.max(np.abs(solver.x_trj[:, 4])) <= np.pi / 4 + 1e-6


def test_profile_descent_reports_phase_times(api):
    """`solver.profile_descent()`: per-phase device times of a descent (the reference has no timing hooks beyond the
    elapsed-time print of iterate, irs_lqr.py:205-208); the solver's state and noise stream position are untouched."""
    cfg = ec.CONFIGS["quadrotor"](T=30)
    s = make_system(api, "quadrotor")
    smp = api.GaussianSampling(cfg["sigma"][:12], cfg["sigma"][12:], 4096, power=cfg["power"], seed=3)
    solver = api.IrsLqrZeroOrder(s, make_params(api, cfg, T=30), smp)
    x0, u0, c0, it0 = solver.x_trj.copy(), solver.u_trj.copy(), solver.cost, solver.iter
    t = solver.profile_descent(repeats=2)
    for key in ("linearize_ms", "riccati_ms", "rollout_ms", "plan_check_ms", "phases_sum_ms", "local_descent_wall_ms"):
        assert key in t and t[key] > 0.0, key
    assert abs(t["phases_sum_ms"] - (t["linearize_ms"] + t["riccati_ms"] + t["rollout_ms"] + t["plan_check_ms"])) < 1e-9
    assert solver.timings is t and solver.iter == it0 and solver.cost == c0
    np.testing.assert_array_equal(solver.x_trj, x0)
    np.testing.assert_array_equal(solver.u_trj, u0)
