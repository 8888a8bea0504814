"""User-written dynamics that read arrays from device memory: CudaSourceDynamics(..., arrays=...) (GPU: -m gpu).

Test systems (oracle/user_arrays.py):
- a linear plant x' = A x + B u + c at (12, 4), A, B and c as arrays, with a float64 numpy twin;
- the reference's pendulum network (tests/golden/mlp_pendulum.npz) written as a source body, ReLU as fmax;
- a 5-64-64-4 tanh cart-pole network, a shape MlpDynamics refuses, with a float64 torch twin;
- a cart whose thrust is a lookup table read at an index computed from its speed.
"""
import concurrent.futures
import ctypes
import gc
import os

import numpy as np
import pytest

from irs_mpc_b200 import _lib, user_system
from oracle import cpu_restatement as cr
from oracle import user_arrays as ua

LIN_NM = (12, 4)
LIN = ua.linear_arrays(*LIN_NM, seed=0)
LIN2 = ua.linear_arrays(*LIN_NM, seed=1)


def golden_weights():
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mlp_pendulum.npz"))
    return [g[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")]


def cartpole_weights():
    return ua.cartpole_net(seed=0)[1]


CARTPOLE_NET_H = 0.05


# name -> (dim_x, dim_u, h, params, step, arrays, autodiff)
def specs():
    return {
        "linear": (12, 4, 0.0, [], ua.LINEAR_STEP, LIN, True),
        "mlp_src": (2, 1, 0.0, [], ua.MLP_STEP, ua.mlp_arrays(golden_weights()), False),
        "mlp_src_ad": (2, 1, 0.0, [], ua.MLP_STEP, ua.mlp_arrays(golden_weights()), True),
        "cartpole_net": (4, 1, CARTPOLE_NET_H, [], ua.RESIDUAL_MLP_STEP, ua.mlp_arrays(cartpole_weights()), True),
        "thrust": (2, 1, ua.THRUST_H, ua.THRUST_PARAMS, ua.THRUST_STEP, {"tab": ua.thrust_table()}, False),
    }


# ------------------------------------------------------------------------------------------------
# CPU: validation, source, hash, compile
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arrays,match", [
    ({"A": [[1.0, 2.0], [3.0, float("nan")]]}, "'A'.*finite"),
    ({"A": [1.0, float("inf")]}, "'A'.*finite"),
    ({"A": np.array([1 + 2j])}, "'A'.*real"),
    ({"A": ["a", "b"]}, "'A'.*real"),
    ({"A": []}, "'A'.*empty"),
    ({"A": np.zeros((2, 0))}, "'A'.*empty"),
    ({"A": 3.0}, "'A'.*0 dimensions"),
    ({"A": np.zeros((1, 1, 1, 1))}, "'A'.*4 dimensions"),
    ({"2A": [1.0]}, "'2A'.*identifier"),
    ({"a-b": [1.0]}, "'a-b'.*identifier"),
    ({"": [1.0]}, "identifier"),
    ({"x": [1.0]}, "'x'.*taken"),
    ({"p": [1.0]}, "'p'.*taken"),
    ({"R": [1.0]}, "'R'.*taken"),
    ({"B": [1.0]}, "'B'.*taken"),
    ({"Math": [1.0]}, "'Math'.*taken"),
    ({"sin": [1.0]}, "'sin'.*taken"),
    ({"int": [1.0]}, "'int'.*taken"),
    ({"template": [1.0]}, "'template'.*taken"),
    ({"irs_table": [1.0]}, "'irs_table'.*prefix"),
    ({"__t": [1.0]}, "'__t'.*prefix"),
    ({"A": [1.0], "A_n0": [1.0]}, "'A_n0'.*extent"),
    ({"A": np.zeros(1 << 23), "Bb": np.zeros((1 << 23) + 1)}, "'Bb'.*limit"),
    ([("A", [1.0])], "mapping"),
])
def test_arrays_are_checked_before_compiling(monkeypatch, arrays, match):
    monkeypatch.setattr(user_system, "_compile", lambda *a: pytest.fail("compiled"))
    with pytest.raises(ValueError, match=match):
        user_system.CudaSourceDynamics(2, 1, 0.05, [], step="o[0] = x[0]; o[1] = x[1] + u[0];", arrays=arrays)
    with pytest.raises(ValueError, match=match):
        user_system.build_library(2, 1, 1, "o[0] = x[0]; o[1] = x[1] + u[0];", arrays=arrays)


def test_set_array_refuses_a_wrong_name_or_shape():
    s = user_system.CudaSourceDynamics.__new__(user_system.CudaSourceDynamics)
    s.system_name, s._arrays = "t", {"A": (0, np.zeros((2, 2)))}
    with pytest.raises(ValueError, match="no array 'Bx'"):
        s.set_array("Bx", np.zeros((2, 2)))
    with pytest.raises(ValueError, match=r"'A' has shape \(2, 2\)"):
        s.set_array("A", np.zeros(4))
    with pytest.raises(ValueError, match="'A'.*finite"):
        s.set_array("A", np.full((2, 2), np.nan))


@pytest.mark.parametrize("autodiff", [False, True])
def test_without_arrays_the_source_is_unchanged(autodiff):
    step = "o[0] = x[0] + h * x[1]; o[1] = x[1] + h * (u[0] - p[0] * x[1]);"
    base = user_system.generate_source(2, 1, 2, step, None, autodiff)
    assert user_system.generate_source(2, 1, 2, step, None, autodiff, arrays=None) == base
    assert user_system.generate_source(2, 1, 2, step, None, autodiff, arrays={}) == base
    assert "user_arrays" not in base and "IRS_USER_ARRAYS" not in base
    assert "#define IRS_USER_NPARAMS 2" in base


def test_source_holds_shapes_not_values():
    step = ua.LINEAR_STEP
    a = user_system.generate_source(12, 4, 1, step, arrays=LIN)
    assert a == user_system.generate_source(12, 4, 1, step, arrays=LIN2)
    other = dict(LIN, c=np.zeros((12, 1)))
    assert a != user_system.generate_source(12, 4, 1, step, arrays=other)
    assert "#define IRS_USER_NPARAMS 2" in a and "#define IRS_USER_ARRAY_ELEMS %d" % (144 + 48 + 12) in a
    assert "%.6f" % LIN["A"][0, 1] not in a


def test_same_shapes_share_a_library_hash(tmp_path, monkeypatch):
    """build_library with the compiler stubbed: same shapes, same hash and path; a new shape, a new hash."""
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    monkeypatch.setattr(user_system, "_nvcc_version", lambda nvcc: "stub nvcc")
    built = []

    def fake_compile(src, out):
        built.append(src)
        with open(out, "wb") as fh:
            fh.write(b"")
    monkeypatch.setattr(user_system, "_compile", fake_compile)
    p1, t1, h1 = user_system.build_library(12, 4, 1, ua.LINEAR_STEP, name="lin", arrays=LIN)
    p2, t2, h2 = user_system.build_library(12, 4, 1, ua.LINEAR_STEP, name="lin", arrays=LIN2)
    assert (p1, h1) == (p2, h2) and t2 == 0.0 and len(built) == 1
    p3, _, h3 = user_system.build_library(12, 4, 1, ua.LINEAR_STEP, name="lin", arrays=dict(LIN, c=np.ones((12, 1))))
    assert h3 != h1 and p3 != p1 and len(built) == 2
    _, _, h4 = user_system.build_library(12, 4, 1, ua.LINEAR_STEP, name="lin")
    assert h4 not in (h1, h3)


VIEW_STEP = """
    R acc = c[0] + T3(1, 0, 1) * T3[T3_n0 * T3_n1 * T3_n2 - 1];
#pragma unroll
    for (int i = 0; i < A_n0; ++i)
#pragma unroll
        for (int j = 0; j < A_n1; ++j) acc += A(i, j) * x[j];
    o[0] = x[0] + h * acc;
    o[1] = x[1] + h * (u[0] * c[c_n0 - 1] - A[0] * x[1]);
"""
VIEW_ARRAYS = {"A": np.eye(2), "c": [1.0, 2.0, 3.0], "T3": np.arange(12.0).reshape(2, 3, 2)}


@pytest.mark.parametrize("autodiff", [False, True])
def test_views_compile_for_sm100a(tmp_path, monkeypatch, autodiff):
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    path, secs, _ = user_system.build_library(2, 1, 1, VIEW_STEP, name="views", autodiff=autodiff,
                                              arrays=VIEW_ARRAYS)
    assert secs > 0 and os.path.getsize(path) > 0
    h = ctypes.CDLL(path)
    for name in ("irs_user_arrays_register", "irs_user_arrays_update", "irs_user_arrays_release"):
        assert hasattr(h, name)


@pytest.mark.parametrize("write,line", [("A[0] = R(1);", 2), ("A(0, 1) += x[0];", 2)])
def test_writing_to_an_array_does_not_compile(tmp_path, monkeypatch, write, line):
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    step = "o[0] = x[0];\n%s\no[1] = x[1] + u[0];\n" % write
    with pytest.raises(RuntimeError, match=r"step\(%d\)" % line):
        user_system.build_library(2, 1, 1, step, name="writes", arrays={"A": np.eye(2)})


def test_main_library_refuses_array_sets(built_lib):
    h = ctypes.c_int(-1)
    v = (ctypes.c_double * 2)(1.0, 2.0)
    vp = ctypes.cast(v, ctypes.c_void_p)
    assert built_lib.irs_user_arrays_register(vp, 2, ctypes.byref(h)) != 0
    assert b"user-written system" in built_lib.irs_last_error()
    assert built_lib.irs_user_arrays_update(0, 0, vp, 2, None) != 0
    assert built_lib.irs_user_arrays_release(0) != 0


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def built():
    """Every library of this module, compiled in parallel (or found in the user cache)."""
    with concurrent.futures.ThreadPoolExecutor(8) as pool:
        futs = {name: pool.submit(user_system.build_library, n, m, 1 + len(prm), step, None, name, ad, arr)
                for name, (n, m, h, prm, step, arr, ad) in specs().items()}
        futs["linear_literal"] = pool.submit(user_system.build_library, 12, 4, 1, ua.linear_literal_step(LIN),
                                             None, "linear_literal", True)
        return {name: f.result() for name, f in futs.items()}


def make(built, name, arrays=None):
    n, m, h, prm, step, arr, ad = specs()[name]
    s = user_system.CudaSourceDynamics(n, m, h, prm, step=step, autodiff=ad, name=name,
                                       arrays=arr if arrays is None else arrays)
    assert s.library_path == built[name][0]
    return s


_SYSTEMS = {}


def system(built, name):
    if name not in _SYSTEMS:
        _SYSTEMS[name] = make(built, name)
    return _SYSTEMS[name]


@pytest.fixture(scope="module")
def api():
    import irs_mpc_b200.all as a
    return a


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


def linear_cfg(T):
    n, m = LIN_NM
    return dict(T=T, Q=np.eye(n), Qd=10.0 * np.eye(n), R=0.1 * np.eye(m), x0=0.5 * np.ones(n),
                xd_trj=np.tile(np.linspace(-1.0, 1.0, n), (T + 1, 1)), u_trj_initial=np.zeros((T, m)),
                sigma=0.05 * np.ones(n + m))


def cartpole_cfg(T):
    return dict(T=T, Q=np.diag([1.0, 1.0, 0.1, 0.1]), Qd=np.diag([50.0, 50.0, 5.0, 5.0]), R=np.diag([0.1]),
                x0=np.zeros(4), xd_trj=np.tile([0.5, -0.3, 0.0, 0.0], (T + 1, 1)), u_trj_initial=np.zeros((T, 1)),
                sigma=np.array([0.05, 0.05, 0.1, 0.1, 0.5]))


def params_of(api, cfg):
    p = api.IrsLqrParameters()
    for key in ("Q", "Qd", "R", "x0", "xd_trj", "u_trj_initial"):
        setattr(p, key, cfg[key])
    for key in ("xbound", "ubound"):
        setattr(p, key, cfg.get(key))
    return p


def sampler_of(api, cfg, N, seed):
    n = cfg["Q"].shape[0]
    return api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, seed=seed)


# ------------------------------------------------------------------------------------------------
# 1. linear plant at (12, 4)
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_linear_plant_dynamics_and_exact_linearization(built, api):
    import torch
    s, twin = system(built, "linear"), ua.LinearTwin(LIN)
    rng = np.random.default_rng(3)
    x, u = rng.standard_normal((1000, 12)), rng.standard_normal((1000, 4))
    assert rel(s.dynamics_batch(x, u), twin.dynamics_batch(x, u)) <= 1e-12
    assert rel(s.dynamics(x[5], u[5]), twin.dynamics(x[5], u[5])) <= 1e-12
    # fp32: the fp32 copy of the arrays (rounded once from float64)
    x32, u32 = x.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)
    assert rel(s._run_dynamics(x32, u32, True, dtype=torch.float32), twin.dynamics_batch(x32, u32)) <= 1e-5
    J = s.jacobian_xu_batch(x[:50], u[:50])
    assert rel(J, twin.jacobian_xu_batch(x[:50], u[:50])) <= 1e-12
    cfg = linear_cfg(20)
    exact = api.IrsLqrExact(s, params_of(api, cfg))
    At, Bt, ct = exact.get_TV_matrices(exact.x_trj, exact.u_trj)
    AB = np.concatenate((At, Bt), axis=2)
    assert np.max(np.abs(AB - np.hstack((LIN["A"], LIN["Bu"]))[None])) <= 1e-12
    assert np.max(np.abs(ct - LIN["c"][None])) <= 1e-12


@pytest.mark.gpu
def test_linear_plant_zero_order_partials(built):
    import test_user_dims_kernels as tdk
    s = system(built, "linear")
    with tdk.engine(s, 1):
        for N in (1, 257, 4097):
            for anti in (False, True):
                _, err = tdk.run_zero_order(s, LIN_NM, N, 3, 1, anti)
                assert err <= user_system_tol_tc()


def user_system_tol_tc():
    from oracle import sample_gram as sg
    return sg.TOL_TENSOR_CORES


@pytest.mark.gpu
def test_linear_plant_first_order_means(built):
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    from oracle import sample_gram as sg
    n, m = LIN_NM
    s = system(built, "linear")
    P = 3
    rng = np.random.default_rng(5)
    x_nom, u_nom = rng.standard_normal((P, n)), rng.standard_normal((P, m))
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    sig = 0.05 * np.ones(n + m)
    for N in (1, 129, 4097):
        sampler = sampling.GaussianSampling(sig[:n], sig[n:], N, seed=21)
        ws = tsk.guarded_workspace(s, smoothing.FIRST_ORDER, P, N)
        smoothing.accumulate(s, smoothing.FIRST_ORDER, xd, ud, N, ws, sigma=sampler.sigma(2), seed=21, it=2,
                             flags=sampler.flags())
        At, Bt, _, status = smoothing.finalize(s, smoothing.FIRST_ORDER, xd, ud, ws, N)
        torch.cuda.synchronize()
        tsk.check_guard(ws)
        assert int(status.sum().item()) == 0
        AB = np.concatenate((_device.to_numpy(At), _device.to_numpy(Bt)), axis=2)
        for p in range(P):
            z = sampler.deltas(1, 2, t0=p)[0]
            pts = (np.concatenate((x_nom[p], u_nom[p])).astype(np.float32)[None, :] + z).astype(np.float32)
            J = s.jacobian_xu_batch(pts[:, :n], pts[:, n:], dtype=torch.float32)
            mean, scale = J.mean(axis=0), np.abs(J).mean(axis=0)
            err = np.abs(AB[p] - mean)
            assert np.all(err[scale == 0] == 0)
            assert float(np.max(err[scale > 0] / scale[scale > 0])) < sg.TOL_CUDA_CORES
            # and the mean of a constant Jacobian is the fp32 copy of [A | B]
            assert np.max(np.abs(AB[p] - np.hstack((LIN["A"], LIN["Bu"])))) < 1e-6


@pytest.mark.gpu
def test_linear_plant_bounded_descent_first_qp_is_certified(built, api):
    from oracle import box_kkt as bk
    from irs_mpc_b200 import _device
    from irs_mpc_b200.tv_lqr import box_solve_device
    T = 20
    cfg = linear_cfg(T)
    ub = np.array([-0.3 * np.ones(4), 0.3 * np.ones(4)])
    cfg["ubound"] = ub
    s = system(built, "linear")
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler_of(api, cfg, 3000, 6))
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    big = 1e30 * np.ones(12)
    dev = [_device.to_device(v[None]) for v in (At, Bt, ct)]
    xq, uq, _, status, _ = box_solve_device(
        s, False, *dev, solver._dQ, solver._dQd, solver._dR, cfg["Q"], cfg["Qd"], cfg["R"], solver._dxd, 0,
        _device.to_device(cfg["x0"][None]), -big, big, ub[0], ub[1])
    assert int(status.item()) == 0
    uq = _device.to_numpy(uq[0])
    qp = bk.BoxQP(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], -big, big, ub[0], ub[1])
    c = qp.certify(uq)
    assert c["certified"], (c["min_lam"], c["max_violation"], c["kkt_residual"])
    assert np.any(np.abs(np.abs(uq) - 0.3) < 1e-6)
    solver2 = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler_of(api, cfg, 3000, 6))
    x_new, u_new = solver2.local_descent(solver2.x_trj, solver2.u_trj)
    assert solver2.bounded_admm_iterations > 0
    assert np.max(np.abs(u_new[0] - uq[0])) < 1e-6 and np.all(np.abs(u_new) <= 0.3 + 1e-6)


# ------------------------------------------------------------------------------------------------
# 2. the reference's pendulum network as a source body
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_pendulum_network_as_source_matches_the_oracle_and_the_reference(built, api):
    from oracle import example_configs as ec
    from oracle.mlp_ref import MlpOracle
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mlp_pendulum.npz"))
    s = system(built, "mlp_src")
    orc = MlpOracle(golden_weights())
    pts = g["pts"]
    assert rel(s.dynamics_batch(pts[:, :2], pts[:, 2:]), orc.dynamics_batch(pts[:, :2], pts[:, 2:])) < 1e-5
    assert rel(s.dynamics_batch(pts[:, :2], pts[:, 2:]), g["out"]) < 1e-5
    T, N, d = g["noise_shape"]
    noise = np.random.default_rng(int(g["noise_seed"])).standard_normal((T, N, d)).astype(np.float32)
    state = {"t": 0}

    def sampling(xbar, ubar, it):
        e = noise[state["t"] % T].astype(np.float64)
        state["t"] += 1
        return e[:, :2], e[:, 2:]
    cfg = ec.pendulum_nn(T=int(T))
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampling)
    At, Bt, ct = solver.get_TV_matrices(g["x_trj"], g["u_trj"])
    assert rel(At, g["At"]) < 1e-4 and rel(Bt, g["Bt"]) < 1e-4 and rel(ct, g["ct"]) < 1e-4


@pytest.mark.gpu
def test_pendulum_network_autodiff_matches_torch_autograd(built):
    import torch
    s = system(built, "mlp_src_ad")
    W1, b1, W2, b2, W3, b3 = [torch.from_numpy(np.asarray(w, dtype=np.float64)) for w in golden_weights()]

    def net(xu):
        return torch.relu(torch.relu(xu @ W1.T + b1) @ W2.T + b2) @ W3.T + b3
    rng = np.random.default_rng(8)
    xu = 2.0 * rng.standard_normal((200, 3))
    J = s.jacobian_xu_batch(xu[:, :2], xu[:, 2:])
    want = np.stack([torch.autograd.functional.jacobian(net, torch.from_numpy(r)).numpy() for r in xu])
    assert np.max(np.abs(J - want)) <= 1e-12 * max(1.0, float(np.abs(want).max()))
    assert rel(s.dynamics_batch(xu[:, :2], xu[:, 2:]), net(torch.from_numpy(xu)).numpy()) <= 1e-12


# ------------------------------------------------------------------------------------------------
# 3. a cart-pole network 5-64-64-4 with tanh
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cartpole_network_matches_torch(built, api):
    import torch
    s = system(built, "cartpole_net")
    net = ua.cartpole_net(seed=0)[0]
    rng = np.random.default_rng(9)
    x, u = rng.standard_normal((300, 4)), rng.standard_normal((300, 1))
    xu = torch.from_numpy(np.hstack((x, u)))
    def step(r):
        r2 = r.reshape(-1, 5)
        return (r2[:, :4] + CARTPOLE_NET_H * (torch.stack(ua.residual_drive(r2[:, :4], r2[:, 4:]), 1) + net(r2))
                ).reshape(r.shape[:-1] + (4,))
    with torch.no_grad():
        want = step(xu).numpy()
    assert rel(s.dynamics_batch(x, u), want) <= 1e-12
    assert rel(ua.MlpTwin(cartpole_weights(), 4, 1, act="tanh", h=CARTPOLE_NET_H).dynamics_batch(x, u), want) <= 1e-12
    J = s.jacobian_xu_batch(x[:60], u[:60])

    Jw = np.stack([torch.autograd.functional.jacobian(step, xu[i]).numpy() for i in range(60)])
    assert np.max(np.abs(J - Jw)) <= 1e-12 * max(1.0, float(np.abs(Jw).max()))


@pytest.mark.gpu
@pytest.mark.parametrize("solver_name", ["IrsLqrExact", "IrsLqrFirstOrder"])
def test_cartpole_network_descents_lower_the_cost(built, api, solver_name):
    cfg = cartpole_cfg(30)
    s = system(built, "cartpole_net")
    if solver_name == "IrsLqrExact":
        solver = api.IrsLqrExact(s, params_of(api, cfg))
    else:
        solver = api.IrsLqrFirstOrder(s, params_of(api, cfg), sampler_of(api, cfg, 2000, 4))
    solver.iterate(4, verbose=False)
    assert solver.cost_lst[-1] < solver.cost_lst[0]


# ------------------------------------------------------------------------------------------------
# 4. a lookup table read at data-dependent indices
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_thrust_table_dynamics_and_partials(built, api):
    import torch
    import test_user_dims_kernels as tdk
    from oracle import sample_gram as sg
    s, twin = system(built, "thrust"), ua.ThrustTwin(ua.thrust_table())
    rng = np.random.default_rng(10)
    x = np.stack((rng.standard_normal(2000), rng.uniform(-3.5, 3.5, 2000)), 1)
    u = rng.standard_normal((2000, 1))
    assert rel(s.dynamics_batch(x, u), twin.dynamics_batch(x, u)) <= 1e-12
    x32, u32 = x.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)
    assert rel(s._run_dynamics(x32, u32, True, dtype=torch.float32), twin.dynamics_batch(x32, u32)) <= 1e-5
    for eng in (0, 1):
        with tdk.engine(s, eng):
            for N in (257, 4097):
                _, err = tdk.run_zero_order(s, (2, 1), N, 3, eng, True, sigma=np.array([0.1, 0.6, 0.3]))
                assert err <= (sg.TOL_TENSOR_CORES if eng else sg.TOL_CUDA_CORES)
    # the fit on the kernel's own deltas against the twin's fit on the same deltas
    T, N = 30, 4000
    cfg = dict(T=T, Q=np.eye(2), Qd=10 * np.eye(2), R=0.1 * np.eye(1), x0=np.array([0.0, -2.0]),
               xd_trj=np.tile([1.0, 1.0], (T + 1, 1)), u_trj_initial=np.ones((T, 1)), sigma=np.array([0.05, 0.3, 0.2]))
    sampler = sampler_of(api, cfg, N, 3)
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler)
    assert rel(solver.x_trj, cr.rollout(twin, cfg["x0"], cfg["u_trj_initial"])) <= 1e-12
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    At_o, Bt_o, ct_o = cr.zero_order_tv_matrices(twin, solver.x_trj, solver.u_trj, deltas)
    assert rel(At, At_o) < 1e-4 and rel(Bt, Bt_o) < 1e-4 and float(np.max(np.abs(ct - ct_o))) < 1e-4


# ------------------------------------------------------------------------------------------------
# 5. set_array
# ------------------------------------------------------------------------------------------------
def _descents(api, s, cfg, k, seed=12):
    solver = api.IrsLqrZeroOrder(s, params_of(api, cfg), sampler_of(api, cfg, 3000, seed))
    return solver, [solver.local_descent(solver.x_trj, solver.u_trj) for _ in range(k)]


@pytest.mark.gpu
def test_set_array_reaches_eager_and_replayed_calls(built, api, monkeypatch):
    from irs_mpc_b200 import _graph
    cfg = linear_cfg(25)
    s1 = make(built, "linear")
    monkeypatch.setattr(user_system, "_compile", lambda *a: pytest.fail("compiled"))
    s2 = make(built, "linear", arrays=LIN2)
    assert s2.cache_hit and s2.source_hash == s1.source_hash and s2.device_params() != s1.device_params()
    solver = api.IrsLqrZeroOrder(s1, params_of(api, cfg), sampler_of(api, cfg, 3000, 12))
    for _ in range(4):
        solver.local_descent(solver.x_trj, solver.u_trj)      # captured on the third call
    graph = solver._graphs._slots["descent"][1]
    assert graph is not None
    for name in ("A", "Bu", "c"):
        s1.set_array(name, LIN2[name])
    monkeypatch.setattr(_graph, "USE_GRAPHS", False)
    ref, fresh = _descents(api, s2, cfg, 1)
    _, eager = _descents(api, s1, cfg, 1)
    monkeypatch.setattr(_graph, "USE_GRAPHS", True)
    # the nominal trajectory of the new values (solver's own was rolled out with the old ones)
    after = [solver.local_descent(ref.x_trj, ref.u_trj) for _ in range(3)]
    assert solver._graphs._slots["descent"][1] is graph          # replayed, not re-captured
    for xa, xb in [(r[0], fresh[0][0]) for r in after + eager] + [(r[1], fresh[0][1]) for r in after + eager]:
        assert np.array_equal(xa, xb)
    rng = np.random.default_rng(1)
    x, u = rng.standard_normal((100, 12)), rng.standard_normal((100, 4))
    assert np.array_equal(s1.dynamics_batch(x, u), s2.dynamics_batch(x, u))
    assert np.array_equal(s1.arrays["A"], LIN2["A"])


# ------------------------------------------------------------------------------------------------
# 6. two systems, same source, different values
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_systems_with_the_same_source_keep_apart(built, api, monkeypatch):
    from irs_mpc_b200 import _graph
    cfg = linear_cfg(25)
    sa, sb = make(built, "linear", arrays=LIN), make(built, "linear", arrays=LIN2)
    assert sa.library_path == sb.library_path and sa._array_handle != sb._array_handle
    monkeypatch.setattr(_graph, "USE_GRAPHS", False)
    own = [_descents(api, s, cfg, 1)[1][0] for s in (sa, sb)]
    assert not np.array_equal(own[0][0], own[1][0])
    monkeypatch.setattr(_graph, "USE_GRAPHS", True)
    va = api.IrsLqrZeroOrder(sa, params_of(api, cfg), sampler_of(api, cfg, 3000, 12))
    vb = api.IrsLqrZeroOrder(sb, params_of(api, cfg), sampler_of(api, cfg, 3000, 12))
    for _ in range(5):                                           # replayed from the third call on
        for i, v in enumerate((va, vb)):
            x, u = v.local_descent(v.x_trj, v.u_trj)
            assert np.array_equal(x, own[i][0]) and np.array_equal(u, own[i][1])
    assert va._graphs._slots["descent"][1] is not None and vb._graphs._slots["descent"][1] is not None
    del vb, sb
    gc.collect()
    for _ in range(2):
        x, u = va.local_descent(va.x_trj, va.u_trj)
        assert np.array_equal(x, own[0][0]) and np.array_equal(u, own[0][1])


# ------------------------------------------------------------------------------------------------
# 7. every other path an arrays system reaches
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_batched_instances_and_cem(built, api):
    T, I = 25, 6
    cfg = cartpole_cfg(T)
    s = system(built, "cartpole_net")
    x0 = np.random.default_rng(2).standard_normal((I, 4)) * 0.1
    xd = np.broadcast_to(cfg["xd_trj"], (I, T + 1, 4)).copy()

    def run(lo, hi):
        bat = api.BatchedIrsLqrZeroOrder(s, cfg["Q"], cfg["Qd"], cfg["R"], x0[lo:hi], xd[lo:hi],
                                         cfg["u_trj_initial"], sampler_of(api, cfg, 2000, 8), instance_offset=lo)
        return bat.iterate(2)
    full, part = run(0, I), run(2, 5)
    for a, b in zip(full, part):
        assert np.array_equal(a[2:5], b)
    twin = ua.MlpTwin(cartpole_weights(), 4, 1, act="tanh", h=CARTPOLE_NET_H)
    p = api.CemParameters()
    p.Q, p.Qd, p.R, p.x0, p.xd_trj, p.u_trj_initial = (cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"],
                                                       cfg["u_trj_initial"])
    B = 64
    p.n_elite, p.batch_size, p.initial_std = 8, B, 0.5 * np.ones(1)
    np.random.seed(99)
    cem = api.CrossEntropyMethod(s, p)
    x_new, u_new = cem.local_descent(cem.x_trj, cem.u_trj)
    np.random.seed(99)
    cand = np.random.normal(cfg["u_trj_initial"], np.tile(p.initial_std, (T, 1)), (B, T, 1))
    costs = np.array([cr.evaluate_cost(cr.rollout(twin, cfg["x0"], cand[k]), cand[k], cfg["xd_trj"], cfg["Q"],
                                       cfg["R"]) for k in range(B)])
    u_o = cand[np.argpartition(costs, p.n_elite)[:p.n_elite]].mean(axis=0)
    np.testing.assert_allclose(u_new, u_o, rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(x_new, cr.rollout(twin, cfg["x0"], u_o), rtol=1e-9, atol=1e-9)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["zero_order_AB", "first_order", "exact"])
def test_worker_modes(built, mode):
    from irs_mpc_b200 import worker
    s = system(built, "linear")
    rng = np.random.default_rng(4)
    x, u = rng.standard_normal((7, 12)), rng.standard_normal((7, 4))
    AB = worker.GpuLinearizationWorker(s, mode=mode, std_x=0.05, seed=3).calc_AB_batch(x, u, 2000, 0.05)
    want = np.hstack((LIN["A"], LIN["Bu"]))
    tol = {"exact": 1e-12, "first_order": 1e-6, "zero_order_AB": 1e-3}[mode]
    assert np.max(np.abs(AB - want[None])) < tol, mode
