"""The rollout kernels of the four built-in systems and the cross-entropy-method elite step, against float64 references
of the same operation (GPU tests: run with `-m gpu`; the refusals and the checks of the references run without one).

A rollout is the forward pass of every iRS-LQR descent, of BatchedIrsLqr* and of CEM: x_{t+1} = f(x_t, u_t) with
u_t = K_t x_t + k_t (closed loop) or given u_t (open loop), then the cost of IrsLqr.evaluate_cost, whose terminal term
uses Q.  Whole-descent tests see these kernels only through loose tolerances; here every launch is compared with the
float64 oracle (oracle/cpu_restatement.py) instance by instance, at
- I in {1, 2, 3, 65}: one instance, both warps of one block, an idle second warp in the last block, many blocks;
- T in {1, 2, 33, 60}: no prefetch, one prefetch, and cost lanes that wrap (t = lane + 32);
- targets per instance (xd_stride = (T + 1) n) and shared (xd_stride = 0);
- dense, non-diagonal Q and R.  They are symmetric: a quadratic form cannot see a transposed weight, so these tests
  do not pin the orientation of Q or R (test_lqr_kernels.py does, for the Riccati kernels).
Every output buffer is filled with NaN before the launch, so a skipped store fails.

Which test reaches which instantiation (Sys<double>, CLOSED = closed / open):

| instantiation                                       | reached by                                                 |
|-----------------------------------------------------|------------------------------------------------------------|
| rollout_kernel<Pendulum / Bicycle / ThreeCart, *>   | test_rollouts_and_costs,                                   |
|                                                     |   test_nan_gain_stays_in_its_instance,                     |
|                                                     |   (ThreeCart) test_three_cart_contact_cases                |
| rollout_kernel<Quadrotor, *>                        | test_rollouts_and_costs [IRS_ROLLOUT_TRIG=0],              |
|                                                     |   test_quadrotor_dispatch [I = 2 SMs + 1, forced 0]        |
| rollout_trig_kernel<Quadrotor, *>                   | test_rollouts_and_costs [IRS_ROLLOUT_TRIG=1],              |
|                                                     |   test_quadrotor_dispatch [I = 2 SMs, forced 1]            |
| warp_trajectory_cost<n, m> inside each of them      | every rollout test                                         |
| cem_rank_kernel, cem_refit_kernel                   | test_cem_elites_and_refit                                  |
| the host checks of irs_cem_refit                    | test_cem_refit_refusals (no GPU)                           |

Properties beyond the oracle: the open-loop rollout of the inputs a closed loop returns replays its trajectory and cost
bit for bit (test_rollouts_and_costs); NaN in one instance's gains leaves every other instance bit-identical
(test_nan_gain_stays_in_its_instance); the quadrotor's default kernel choice is observed on both sides of I = 2 SMs
(test_quadrotor_dispatch).

The references are vectorised over instances (`reference`); test_reference_is_the_scalar_oracle shows on the CPU that
they are cr.closed_loop_descent / cr.rollout row by row.  three_cart steps with the scalar semantics
(dynamics_scalar_batch: half-depth push-out), as the rollouts do.  An instance whose oracle free step passes within
CONTACT_MARGIN of a contact threshold is left out: the GPU's FMA contraction may legitimately put it in the other case.

CEM: the elite mask must be exactly the first n_elite indices of np.argsort(cost, kind="stable"), the order of the key
(isnan(cost), cost, index) (NaN after +inf, ties by index), for B across the 256-wide rank tiles and cost patterns with
ties, signed zeros, infinities and NaN; mean and population std (ddof = 0) over those elites against numpy float64 at
1e-13 of max |u|, for widths T m across the 128-wide refit block.

Tolerance of the rollouts: 1e-12 relative (max-abs error over max-abs value, per instance) for trajectories and inputs,
and for each cost, as for the user-written systems (test_user_dims_kernels.py: test_rollouts_and_costs).  One ulp of
relative noise injected into every input and state of the float64 references, every step, grows over T = 100 to at
most 9e-15 for pendulum, bicycle and three_cart and 7e-14 for the quadrotor's closed loop, but to 1.4e-12 for its
open loop: a hovering quadrotor without feedback integrates a perturbation of its body rates three times before it
reaches the position.  The GPU differs from numpy in only a few operations per step (sincos, FMA contraction), and
its measured error (below) stays under that bound.  The quadrotor's gains carry an attitude-damping term (`attitude_damping`), and its
open-loop inputs are those of a second damped closed loop: with random gains of 1e-3 alone the attitude is a random
walk, some of 297 instances tumble within T = 60, and one-ulp noise in the others grows past 1e-12.

Largest errors measured on a B200 (1000 W power limit), relative as above:

| system     | closed-loop x, u | closed-loop cost | open-loop x | open-loop cost |
|------------|------------------|------------------|-------------|----------------|
| pendulum   | 6.7e-15          | 1.1e-15          | 1.2e-15     | 9.8e-16        |
| bicycle    | 1.7e-15          | 1.0e-15          | 8.1e-16     | 8.1e-16        |
| quadrotor  | 8.7e-14          | 7.3e-15          | 2.9e-13     | 5.7e-14        |
| three_cart | 7.6e-16          | 8.5e-16          | 7.6e-16     | 9.1e-16        |

CEM mean and std: 2.7e-17 and 4.3e-16 of max |u|.  The largest error of every check is printed at the end of the
module (-s shows it).
"""
import ctypes

import numpy as np
import pytest

from oracle import cpu_restatement as cr
from oracle import example_configs as ec

SYSTEMS = ["pendulum", "bicycle", "quadrotor", "three_cart"]
CLASSES = {"pendulum": "PendulumDynamics", "bicycle": "BicycleDynamics", "quadrotor": "QuadrotorDynamics",
           "three_cart": "ThreeCartDynamics"}
INSTANCES = [1, 2, 3, 65]
HORIZONS = [1, 2, 33, 60]
RTOL = 1e-12
CONTACT_MARGIN = 1e-9
# spread of the random parts: gains, inputs around the configuration's initial inputs, initial state around its x0
SPREAD = {"pendulum": (0.1, 0.5, 0.5), "bicycle": (0.05, 0.3, 0.3), "quadrotor": (1e-3, 0.02, 0.05),
          "three_cart": (0.1, 1.0, 0.05)}
CEM_B = [1, 2, 255, 256, 257, 1000, 4097]
CEM_PATTERNS = ["distinct", "ties", "signed_zeros", "infinities", "nan_before_inf", "all_nan"]
CEM_WIDTHS = [(1, 1), (127, 1), (32, 4), (43, 3), (100, 4)]          # T m = 1, 127, 128, 129, 400
CEM_RTOL = 1e-13
MAX_ERR = {}


def note(key, v):
    MAX_ERR[key] = max(MAX_ERR.get(key, 0.0), float(v))


@pytest.fixture(scope="module", autouse=True)
def report_max_errors():
    yield
    for k, v in sorted(MAX_ERR.items()):
        print("\nlargest %s: %.3e" % (k, v))


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


# ------------------------------------------------------------------------------------------------
# problems and float64 references
# ------------------------------------------------------------------------------------------------
def attitude_damping(orc):
    """Gains [m, n] of a PD loop on roll, pitch and yaw (natural frequency 4 rad/s, damping 0.7 in every axis):
    the rotor commands that produce the moment -(kp angle + kd rate) about each body axis."""
    K = np.zeros((orc.dim_u, orc.dim_x))
    signs = np.array([[-1., -1, 1, 1], [-1., 1, 1, -1], [-1., 1, -1, 1]])     # moment of each rotor per axis
    arm = np.array([orc.L * orc.kF, orc.L * orc.kF, orc.kM])
    w, zeta = 4.0, 0.7
    for j in range(3):
        kp, kd = orc.Idiag[j] * w * w, 2.0 * zeta * w * orc.Idiag[j]
        K[:, 3 + j] = -signs[j] * kp / (4.0 * arm[j])
        K[:, 9 + j] = -signs[j] * kd / (4.0 * arm[j])
    return K


def problem(name, I, T, seed):
    """Closed- and open-loop inputs of I instances of the system `name`, shared and per-instance targets, dense
    symmetric positive definite weights.  The quadrotor's open-loop inputs are those of a second damped closed loop
    (random inputs alone would tumble it)."""
    cfg = ec.CONFIGS[name](T=T)
    orc = cr.SYSTEMS[name](cfg["h"])
    n, m = orc.dim_x, orc.dim_u
    ks, us, xs = SPREAD[name]
    rng = np.random.default_rng(seed)
    u_init = cfg["u_trj_initial"][None, :T]

    def gains():
        K = ks * rng.standard_normal((I, T, m, n))
        return K + attitude_damping(orc) if name == "quadrotor" else K, u_init + us * rng.standard_normal((I, T, m))
    (K, k), (K2, k2) = gains(), gains()
    A, B = rng.standard_normal((n, n)), rng.standard_normal((m, m))
    xd = cfg["xd_trj"][:T + 1]
    p = dict(name=name, orc=orc, I=I, T=T, n=n, m=m, K=K, k=k, u=k2, x0=cfg["x0"] + xs * rng.standard_normal((I, n)),
             xd=xd, xd_own=xd + 0.5 * rng.standard_normal((I, T + 1, n)),
             Q=A @ A.T / n + 0.1 * np.eye(n), R=B @ B.T / m + 0.1 * np.eye(m))
    if name == "quadrotor":
        p["u"] = reference(dict(p, K=K2, k=k2), True)[1]
    return p


def reference(p, closed):
    """cr.closed_loop_descent (closed) or cr.rollout of every instance at once -> (x [I, T+1, n], u [I, T, m])."""
    orc, I, T = p["orc"], p["I"], p["T"]
    step = orc.dynamics_scalar_batch if p["name"] == "three_cart" else orc.dynamics_batch
    x = np.empty((I, T + 1, p["n"]))
    u = np.empty((I, T, p["m"]))
    x[:, 0] = p["x0"]
    for t in range(T):
        if closed:
            u[:, t] = np.stack([p["K"][i, t].dot(x[i, t]) for i in range(I)]) + p["k"][:, t]
        else:
            u[:, t] = p["u"][:, t]
        x[:, t + 1] = step(x[:, t], u[:, t])
    return x, u


def reference_costs(p, x, u, shared):
    xd = [p["xd"] if shared else p["xd_own"][i] for i in range(p["I"])]
    return np.array([cr.evaluate_cost(x[i], u[i], xd[i], p["Q"], p["R"]) for i in range(p["I"])])


def contact_margin(orc, x, u):
    """Per instance, the closest any free step of the trajectory comes to a contact threshold, |gap - d|."""
    I, T = u.shape[:2]
    s = orc._free_step(x[:, :T].reshape(I * T, -1), u.reshape(I * T, -1))
    gaps = np.stack((s[:, 1] - s[:, 0], s[:, 2] - s[:, 1]), axis=1)
    return np.abs(gaps - orc.d).reshape(I, -1).min(axis=1)


def kept(p, trajectories):
    """Instances compared with the oracle: all but the three_cart ones near a contact threshold (at least 90 %)."""
    keep = np.ones(p["I"], bool)
    if p["name"] == "three_cart":
        for x, u in trajectories:
            keep &= contact_margin(p["orc"], x, u) > CONTACT_MARGIN
        assert keep.mean() >= 0.9, keep
    return keep


@pytest.mark.parametrize("name", SYSTEMS)
def test_reference_is_the_scalar_oracle(name):
    """The vectorised references equal cr.closed_loop_descent / cr.rollout instance by instance."""
    p = problem(name, 3, 33, 5)
    for closed in (True, False):
        x, u = reference(p, closed)
        for i in range(p["I"]):
            if closed:
                xo, uo = cr.closed_loop_descent(p["orc"], p["K"][i], p["k"][i], p["x0"][i])
                assert rel(u[i], uo) <= 1e-14
            else:
                xo = cr.rollout(p["orc"], p["x0"][i], p["u"][i])
            assert np.all(np.isfinite(xo)) and rel(x[i], xo) <= 1e-14, (closed, i)


# ------------------------------------------------------------------------------------------------
# GPU rollouts
# ------------------------------------------------------------------------------------------------
def device_system(name):
    from irs_mpc_b200 import systems
    return getattr(systems, CLASSES[name])(ec.CONFIGS[name]()["h"])


def upload(p):
    from irs_mpc_b200 import _device
    return {key: _device.to_device(p[key]) for key in ("K", "k", "u", "x0", "xd", "xd_own", "Q", "R")}


def launch(p, d, shared, K=None, u=None):
    """irs_rollout_closed_loop with gains K (default d["K"]) and d["k"], or irs_rollout_open_loop of the device inputs
    u, into NaN-filled buffers -> (x_trj, u_trj (closed loop) or None, cost) as device tensors."""
    from irs_mpc_b200 import _device, _lib
    s = device_system(p["name"])
    I, T, n, m = p["I"], p["T"], p["n"], p["m"]
    xd, stride = (d["xd"], 0) if shared else (d["xd_own"], (T + 1) * n)
    xs, cost = _device.empty((I, T + 1, n)).fill_(np.nan), _device.empty((I,)).fill_(np.nan)
    prm, nprm = s._params()
    if u is None:
        K = d["K"] if K is None else K
        us = _device.empty((I, T, m)).fill_(np.nan)
        _lib.call("irs_rollout_closed_loop", s.system_id, prm, nprm, _device.ptr(K), _device.ptr(d["k"]),
                  _device.ptr(d["x0"]), _device.ptr(xd), stride, _device.ptr(d["Q"]), _device.ptr(d["R"]), I, T,
                  _device.ptr(xs), _device.ptr(us), _device.ptr(cost), _device.stream_ptr())
    else:
        us = None
        _lib.call("irs_rollout_open_loop", s.system_id, prm, nprm, _device.ptr(u), _device.ptr(d["x0"]),
                  _device.ptr(xd), stride, _device.ptr(d["Q"]), _device.ptr(d["R"]), I, T, _device.ptr(xs),
                  _device.ptr(cost), _device.stream_ptr())
    return xs, us, cost


def check(p, got, want_x, want_u, want_cost, keep, what):
    from irs_mpc_b200 import _device
    x, c = _device.to_numpy(got[0]), _device.to_numpy(got[2])
    u = None if got[1] is None else _device.to_numpy(got[1])
    for i in np.flatnonzero(keep):
        e = rel(x[i], want_x[i])
        if u is not None:
            e = max(e, rel(u[i], want_u[i]))
        assert e <= RTOL, (what, i, e)
        note("%s %s trajectory error (rel.)" % (p["name"], what), e)
        ec_ = abs(c[i] - want_cost[i]) / abs(want_cost[i])
        assert ec_ <= RTOL, (what, i, c[i], want_cost[i])
        note("%s %s cost error (rel.)" % (p["name"], what), ec_)


def set_trig(monkeypatch, flag):
    if flag is None:
        monkeypatch.delenv("IRS_ROLLOUT_TRIG", raising=False)
    else:
        monkeypatch.setenv("IRS_ROLLOUT_TRIG", flag)


@pytest.mark.gpu
@pytest.mark.parametrize("T", HORIZONS)
@pytest.mark.parametrize("I", INSTANCES)
@pytest.mark.parametrize("name", SYSTEMS)
def test_rollouts_and_costs(name, I, T, monkeypatch):
    """Closed and open loop, shared and per-instance targets, against the oracle; the open-loop rollout of the
    returned inputs replays the closed loop bit for bit.  The quadrotor runs both of its kernels."""
    import torch
    p = problem(name, I, T, 1000 * SYSTEMS.index(name) + 10 * I + T)
    x_c, u_c = reference(p, True)
    x_o, u_o = reference(p, False)
    keep = kept(p, ((x_c, u_c), (x_o, u_o)))
    cost_c = {shared: reference_costs(p, x_c, u_c, shared) for shared in (True, False)}
    cost_o = {shared: reference_costs(p, x_o, u_o, shared) for shared in (True, False)}
    d = upload(p)
    for flag in (["0", "1"] if name == "quadrotor" else [None]):
        set_trig(monkeypatch, flag)
        for shared in (True, False):
            closed = launch(p, d, shared)
            check(p, closed, x_c, u_c, cost_c[shared], keep, "closed-loop")
            replay = launch(p, d, shared, u=closed[1])
            assert torch.equal(replay[0], closed[0]) and torch.equal(replay[2], closed[2]), (flag, shared)
            check(p, launch(p, d, shared, u=d["u"]), x_o, u_o, cost_o[shared], keep, "open-loop")


@pytest.mark.gpu
def test_quadrotor_dispatch(monkeypatch):
    """By default the quadrotor takes rollout_trig_kernel up to I = 2 SMs and rollout_kernel above; both sides of that
    choice, and I = 3 forced each way, against the oracle.  The kernel that ran is read from the profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    T = 60
    for I, flag, kernel in ((2 * sms, None, "rollout_trig_kernel"), (2 * sms + 1, None, "rollout_kernel"),
                            (3, "0", "rollout_kernel"), (3, "1", "rollout_trig_kernel")):
        set_trig(monkeypatch, flag)
        p = problem("quadrotor", I, T, I)
        x_c, u_c = reference(p, True)
        x_o, u_o = reference(p, False)
        for x in (x_c, x_o):
            assert np.all(np.isfinite(x))
            moved = np.max(np.abs(x[:, :, 3:6] - x[:, :1, 3:6]), axis=(1, 2))
            assert np.min(moved) > 1e-3, np.min(moved)                          # every attitude really moved
        keep = np.ones(I, bool)
        d = upload(p)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            closed = launch(p, d, False)
            opened = launch(p, d, True, u=d["u"])
            torch.cuda.synchronize()
        names = [e.key for e in prof.key_averages() if "rollout" in e.key]
        assert names and all(kernel + "<" in k for k in names), (I, flag, names)
        check(p, closed, x_c, u_c, reference_costs(p, x_c, u_c, False), keep, "closed-loop")
        check(p, opened, x_o, u_o, reference_costs(p, x_o, u_o, True), keep, "open-loop")


@pytest.mark.gpu
def test_three_cart_contact_cases():
    """Inputs 1.0 around the configuration's initial ones over T = 100 bring every contact case (all three carts,
    carts 1-2, carts 2-3) into both rollouts."""
    p = problem("three_cart", 20, 100, 77)
    orc, T = p["orc"], p["T"]
    x_c, u_c = reference(p, True)
    x_o, u_o = reference(p, False)
    for x, u in ((x_c, u_c), (x_o, u_o)):
        cases = orc.contact_case(x[:, :T].reshape(-1, 6), u.reshape(-1, 2))
        assert {1, 2, 3} <= set(cases.tolist()), np.bincount(cases)
    keep = kept(p, ((x_c, u_c), (x_o, u_o)))
    d = upload(p)
    for shared in (True, False):
        check(p, launch(p, d, shared), x_c, u_c, reference_costs(p, x_c, u_c, shared), keep, "closed-loop")
        check(p, launch(p, d, shared, u=d["u"]), x_o, u_o, reference_costs(p, x_o, u_o, shared), keep,
              "open-loop")


@pytest.mark.gpu
@pytest.mark.parametrize("name", SYSTEMS)
def test_nan_gain_stays_in_its_instance(name, monkeypatch):
    """NaN in one gain of instance 31 (which shares its block with instance 30) leaves every other instance's
    trajectory, inputs and cost bit-identical, and that instance's steps before it too."""
    import torch
    from irs_mpc_b200 import _device
    I, T, j, t0 = 65, 33, 31, 17
    p = problem(name, I, T, 3 + SYSTEMS.index(name))
    d = upload(p)
    K = p["K"].copy()
    K[j, t0, p["m"] - 1, p["n"] - 1] = np.nan
    dK = _device.to_device(K)
    others = torch.arange(I, device=dK.device) != j
    for flag in (["0", "1"] if name == "quadrotor" else [None]):
        set_trig(monkeypatch, flag)
        base, bad = launch(p, d, False), launch(p, d, False, K=dK)
        for a, b in zip(base, bad):
            assert torch.equal(a[others], b[others]), flag
        assert torch.equal(base[0][j, :t0 + 1], bad[0][j, :t0 + 1]) and torch.equal(base[1][j, :t0], bad[1][j, :t0])
        assert bool(torch.isnan(bad[1][j, t0]).any()) and bool(torch.isnan(bad[2][j]))


# ------------------------------------------------------------------------------------------------
# CEM rank and refit
# ------------------------------------------------------------------------------------------------
def cem_costs(pattern, B, rng):
    if pattern == "distinct":
        return rng.standard_normal(B)
    if pattern == "ties":                                   # small integers: ties straddle every cut
        return rng.integers(0, 4, B).astype(np.float64)
    if pattern == "signed_zeros":                           # -0.0 == +0.0: ties, broken by index
        return rng.choice(np.array([-0.0, 0.0, 0.0, -0.0, -1.0, 1.0]), B)
    if pattern == "infinities":
        return rng.choice(np.array([-np.inf, np.inf, -1.0, 0.5, 2.0]), B)
    if pattern == "nan_before_inf":                         # NaN at the lower indices, +inf above, a few finite
        c = np.full(B, np.inf)
        c[:(B + 1) // 2] = np.nan
        if B > 2:
            few = rng.random(B) < 0.125
            c[few] = rng.standard_normal(int(few.sum()))
        return c
    assert pattern == "all_nan"
    return np.full(B, np.nan)


def stable_elites(cost, n_elite):
    """Mask of the first n_elite indices of the stable argsort: NaN last, ties by index."""
    mask = np.zeros(cost.shape[0], np.int32)
    mask[np.argsort(cost, kind="stable")[:n_elite]] = 1
    return mask


@pytest.mark.gpu
@pytest.mark.parametrize("pattern", CEM_PATTERNS)
@pytest.mark.parametrize("B", CEM_B)
def test_cem_elites_and_refit(B, pattern):
    """irs_cem_refit: the elite mask is exactly the stable-argsort one with n_elite ones; mean and population std
    over those elites against numpy float64."""
    import torch
    from irs_mpc_b200 import _device, _lib
    rng = np.random.default_rng(B * 10 + CEM_PATTERNS.index(pattern))
    cost = cem_costs(pattern, B, rng)
    dcost = _device.to_device(cost)
    for T, m in CEM_WIDTHS:
        u = rng.standard_normal((B, T * m))
        du = _device.to_device(u)
        for n_elite in sorted({v for v in (1, 2, B // 2, B - 1, B) if 1 <= v <= B}):
            elite = _device.empty((B,), torch.int32).fill_(-1)
            mean, std = _device.empty((T * m,)).fill_(np.nan), _device.empty((T * m,)).fill_(np.nan)
            _lib.call("irs_cem_refit", _device.ptr(dcost), _device.ptr(du), B, T, m, n_elite, _device.ptr(elite),
                      _device.ptr(mean), _device.ptr(std), _device.stream_ptr())
            got, want = _device.to_numpy(elite), stable_elites(cost, n_elite)
            assert int(got.sum()) == n_elite and np.array_equal(got, want), (n_elite, T * m, np.flatnonzero(got != want))
            sel = u[want == 1]
            scale = float(np.max(np.abs(u)))
            for key, g, w in (("mean", mean, sel.mean(axis=0)), ("std", std, sel.std(axis=0))):
                e = float(np.max(np.abs(_device.to_numpy(g) - w))) / scale
                assert e <= CEM_RTOL, (key, n_elite, T * m, e)
                note("CEM %s error (units of max |u|)" % key, e)


def test_cem_refit_refusals(built_lib):
    """Host-side checks run before any launch, so they are testable without a GPU: n_elite = 0, n_elite > B, B = 0."""
    buf = (ctypes.c_double * 4)()
    p = ctypes.addressof(buf)              # never read: the call returns before the launch
    for B, n_elite in ((4, 0), (4, 5), (0, 1), (0, 0)):
        rc = built_lib.irs_cem_refit(p, p, B, 1, 1, n_elite, p, p, p, None)
        assert rc != 0 and b"need 1 <= n_elite <= B" in built_lib.irs_last_error(), (B, n_elite)
