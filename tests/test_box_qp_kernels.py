"""Every `box_mpc_kernel<Sys, CACHE>` variant against an exact KKT certificate of the box-constrained QP (run
with `-m gpu`).

Reference: `oracle/box_kkt.py` condenses the QP of irs_lqr/tv_lqr.py:69-137 with its absolute boxes, takes the
active set from the kernel's answer, solves the equality-constrained KKT system on it in float64 and checks
multipliers >= 0 and feasibility of the other rows: the exact minimiser, independent of the ADMM and of its
stopping rule.  Accuracy bar: max |u - u*| and max |x - x*| <= 1e-7 max(1, |.*|_inf).

Which parametrisation reaches which kernel (`launch_box_mpc` in csrc/api.cu: the per-step matrices are staged
in shared memory when `box_mpc_smem_bytes(T, true)` fits in 200 KiB, else CACHE = false; T_max is the longest
horizon whose non-caching layout fits):

| system (id)      | dims    | CACHE = true (T <= T_cache)                        | CACHE = false (T_cache < T <= T_max)           |
|------------------|---------|----------------------------------------------------|------------------------------------------------|
| Pendulum (0)     | (2, 1)  | single QP T = 1, 2, 12, 913; MPC T = 12, 40        | single QP T = 914, 1827                        |
| Bicycle (1)      | (5, 2)  | single QP T = 1, 2, 12, 258; MPC T = 12, 40        | single QP T = 259, 774                         |
| Quadrotor (2)    | (12, 4) | single QP T = 1, 2, 12, 64; MPC T = 12, 40         | single QP T = 65, 335; MPC T = 65              |
| ThreeCart (3)    | (6, 2)  | single QP T = 1, 2, 12, 209; MPC T = 12, 40        | single QP T = 210, 672                         |
| Mlp21 (4)        | (2, 1)  | MPC T = 12, 40; single QP T = 913                  | single QP T = 914                              |

Single QPs (`mpc = 0`) go through `tv_lqr.box_solve_device` with the system of matching dimensions (what
`solve_tvlqr` does through `_DimsOnlySystem`), and through `solve_tvlqr` itself; the learned system's single
QP never evaluates the network and must equal the pendulum's bit for bit.  T_max + 1 is refused.
"""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import box_kkt as bk                  # noqa: E402
from oracle import box_tvlqr as bq                # noqa: E402
from oracle import cpu_restatement as cr          # noqa: E402
from oracle import dense_lqr                      # noqa: E402
from oracle import example_configs as ec          # noqa: E402

DIMS = [(2, 1), (5, 2), (6, 2), (12, 4)]
BAR = 1e-7
SMEM_LIMIT = 200 * 1024


def smem_bytes(n, m, T, cache):
    """box_mpc_smem_bytes of csrc/tvlqr_box.cuh, restated: keep the two in step."""
    d = 3 * (T + 1) * n + 4 * T * m + T * n + (T + 1) * n + 2 * n + n + m
    if cache:
        d += T * (n * n + 2 * n * m + m * m + n + m * n + m)
    return 8 * d


def t_cache(n, m):
    return max(T for T in range(1, 4000) if smem_bytes(n, m, T, True) <= SMEM_LIMIT)


def t_max(n, m):
    return max(T for T in range(1, 4000) if smem_bytes(n, m, T, False) <= SMEM_LIMIT)


def test_layout_boundaries_are_the_documented_ones():
    assert {d: (t_cache(*d), t_max(*d)) for d in DIMS} == {(2, 1): (913, 1827), (5, 2): (258, 774),
                                                           (6, 2): (209, 672), (12, 4): (64, 335)}


class Api:
    def __init__(self):
        import torch
        import irs_mpc_b200.all as m
        from irs_mpc_b200 import _device, _lib, tv_lqr
        self.torch, self.dev, self.lib, self.tv, self.m = torch, _device, _lib, tv_lqr, m

    def up(self, a):
        return self.dev.to_device(np.ascontiguousarray(a, dtype=np.float64))


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    return Api()


@pytest.fixture(scope="module")
def mlp(api, golden_dir):
    import os
    g = np.load(os.path.join(golden_dir, "mlp_pendulum.npz"))
    w = [g[k] for k in ("W1", "b1", "W2", "b2", "W3", "b3")]
    from oracle.mlp_ref import MlpOracle
    return api.m.MlpDynamics([(w[0], w[1]), (w[2], w[3]), (w[4], w[5])]), MlpOracle(w)


def solve(api, p, mpc=False, system=None, scale=1.0, max_iter=None, gains=None, x0=None):
    """box_solve_device on the problem dict of bk.make_problem -> numpy (x, u, cost, status, iters)."""
    n, m, T = p["n"], p["m"], p["T"]
    system = system or api.tv._DimsOnlySystem(n, m)
    Q, Qd, R = scale * p["Q"], scale * p["Qd"], scale * p["R"]
    d = {k: api.up(p[k]) for k in ("At", "Bt", "ct", "xd")}
    kw = {} if max_iter is None else {"max_iter": max_iter}
    if gains is not None:
        kw.update(K0=api.up(gains[0]), k0=api.up(gains[1]))
    out = api.tv.box_solve_device(system, mpc, d["At"], d["Bt"], d["ct"], api.up(Q), api.up(Qd), api.up(R), Q, Qd, R,
                                  d["xd"], 0 if p["shared_xd"] else (T + 1) * n, api.up(p["x0"] if x0 is None else x0),
                                  p["xlo"], p["xhi"], p["ulo"], p["uhi"], **kw)
    return tuple(api.dev.to_numpy(v) for v in out)


def check_instance(p, i, x, u, cost, status, iters, scale=1.0, margins=True):
    """Certificate, accuracy bar, rollout, bounds, cost, status of instance i.  Returns the certificate."""
    where = (p["n"], p["m"], p["T"], i)
    assert status[i] == 0 and iters[i] > 0, where + (status[i], iters[i])
    qp = bk.instance_qp(p, i)
    c = qp.certify(u[i])
    assert c["certified"], where + (c["min_lam"], c["max_violation"], c["kkt_residual"])
    if margins:
        lam_rel, slack_rel = qp.margins(c)
        assert lam_rel >= 1e-8 and slack_rel >= 1e-5, where + ("not strictly complementary", lam_rel, slack_rel)
    assert np.max(np.abs(u[i] - c["u"])) <= BAR * max(1.0, np.max(np.abs(c["u"]))), where
    assert np.max(np.abs(x[i] - c["x"])) <= BAR * max(1.0, np.max(np.abs(c["x"]))), where
    # x is the affine rollout of u
    xr = qp.states(u[i])
    assert np.max(np.abs(x[i] - xr)) <= 1e-12 * max(1.0, np.max(np.abs(xr))), where
    # the boxes, to the bar
    xs = max(1.0, np.max(np.abs(x[i])))
    us = max(1.0, np.max(np.abs(u[i])))
    assert np.all(x[i][1:] >= bk._rows(p["xlo"], p["T"], 1) - BAR * xs), where
    assert np.all(x[i][1:] <= bk._rows(p["xhi"], p["T"], 1) + BAR * xs), where
    assert np.all(u[i] >= bk._rows(p["ulo"], p["T"], 0) - BAR * us), where
    assert np.all(u[i] <= bk._rows(p["uhi"], p["T"], 0) + BAR * us), where
    want = cr.evaluate_cost(x[i], u[i], p["xd"][0 if p["shared_xd"] else i], scale * p["Q"], scale * p["R"])
    assert abs(cost[i] - want) <= 1e-12 * abs(want), where + (cost[i], want)
    return c


# ------------------------------------------------------------------------------------------------
# single QP (mpc = 0)
# ------------------------------------------------------------------------------------------------
def horizon_cases():
    out = []
    for n, m in DIMS:
        for T in (1, 2, 12):
            for box in ("input", "state", "both", "tv", "wide"):
                out.append((n, m, T, box))
        tc = t_cache(n, m)
        out += [(n, m, tc, "input"), (n, m, tc + 1, "input"), (n, m, t_max(n, m), "input")]
    out += [(12, 4, 64, "tv"), (12, 4, 65, "tv")]
    return out


@pytest.mark.parametrize("n,m,T,box", horizon_cases())
def test_single_qp_is_certified(api, n, m, T, box):
    """Three instances, the middle one deep inside the box: an indexing error shows up as one wrong instance."""
    I = 3
    p = bk.make_problem(n, m, T, box, "dense", I=I, inactive=(1,), seed=1000 * n + T)
    x, u, cost, status, iters = solve(api, p)
    n_active = 0
    for i in range(I):
        c = check_instance(p, i, x, u, cost, status, iters)
        if box == "wide" or i == 1:
            assert not np.any(c["active"]), i
        n_active += int(np.sum(c["active"]))
        if box == "wide":
            xs, us = dense_lqr.solve(p["At"][i], p["Bt"][i], p["ct"][i], p["Q"], p["Qd"], p["R"], p["x0"][i], p["xd"][i])
            assert np.max(np.abs(u[i] - us)) <= BAR * max(1.0, np.max(np.abs(us)))
    if box != "wide" and T >= 12:
        assert n_active >= 2, n_active


@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("I", [1, 3, 17])
@pytest.mark.parametrize("n,m", DIMS)
def test_instances_and_shared_targets(api, n, m, I, shared):
    T = 20
    inactive = () if shared else tuple(i for i in (1, 5, 16) if i < I)
    p = bk.make_problem(n, m, T, "both", "nonsym", I=I, inactive=inactive, shared_xd=shared, seed=7 * I + n)
    x, u, cost, status, iters = solve(api, p)
    for i in range(I):
        check_instance(p, i, x, u, cost, status, iters)
    # each instance alone gives the same answer (no cross-talk between warps)
    if I > 1:
        i = I - 1
        q = dict(p, I=1, At=p["At"][i:i + 1], Bt=p["Bt"][i:i + 1], ct=p["ct"][i:i + 1], x0=p["x0"][i:i + 1],
                 xd=p["xd"] if shared else p["xd"][i:i + 1])
        x1, u1, c1, _, it1 = solve(api, q)
        assert np.array_equal(u1[0], u[i]) and np.array_equal(x1[0], x[i]) and it1[0] == iters[i]


@pytest.mark.parametrize("kind", ["diag", "dense", "nonsym"])
@pytest.mark.parametrize("n,m", DIMS)
def test_weights_and_their_scale(api, n, m, kind):
    """The QP and its minimiser do not change under a common scaling of (Q, Qd, R), and neither may the
    solve: bit-identical at 2^+-100 (exact in floating point), 1e-12 at 1e+-30.  Each scaled run gets ten
    times the iterations of the unscaled one."""
    T, I = 12, 3
    p = bk.make_problem(n, m, T, "both", kind, I=I, inactive=(1,), seed=31 * n + len(kind))
    x, u, cost, status, iters = solve(api, p)
    for i in range(I):
        check_instance(p, i, x, u, cost, status, iters)
    cap = 10 * int(iters.max())
    for s in (2.0 ** 100, 2.0 ** -100, 1e30, 1e-30):
        xs, us, cs, sts, its = solve(api, p, scale=s, max_iter=cap)
        assert np.all(sts == 0), (s, sts, its)
        if s in (2.0 ** 100, 2.0 ** -100):
            assert np.array_equal(xs, x) and np.array_equal(us, u) and np.array_equal(its, iters), s
            assert np.array_equal(cs, s * cost), s
        else:
            assert np.max(np.abs(us - u)) <= 1e-12 * max(1.0, np.max(np.abs(u))), s
            assert np.max(np.abs(xs - x)) <= 1e-12 * max(1.0, np.max(np.abs(x))), s
            assert np.all(np.abs(cs - s * cost) <= 1e-12 * np.abs(s * cost)), s


@pytest.mark.parametrize("n,m", DIMS)
def test_too_long_horizon_is_refused_before_launch(api, n, m, monkeypatch):
    T = t_max(n, m) + 1
    p = bk.make_problem(n, m, T, "input", "diag", I=1, seed=n)
    made = []
    empty = api.dev.empty

    def marked(*a, **k):
        t = empty(*a, **k)
        t.fill_(-7)
        made.append(t)
        return t
    monkeypatch.setattr(api.dev, "empty", marked)
    with pytest.raises(api.lib.IrsCudaError, match="too long"):
        solve(api, p)
    api.torch.cuda.synchronize()
    # the last four buffers are the kernel's outputs (x, u, cost, status, iters after the Riccati ones)
    for t in made[-5:]:
        assert bool((t == -7).all())


@pytest.mark.parametrize("T", [913, 914])
def test_learned_system_single_qp_equals_the_pendulum(api, mlp, T):
    """The Mlp21 instantiation, both layouts: a single QP never evaluates the dynamics."""
    p = bk.make_problem(2, 1, T, "input", "dense", I=2, seed=T)
    a = solve(api, p)
    b = solve(api, p, system=mlp[0])
    for va, vb in zip(a, b):
        assert np.array_equal(va, vb)
    check_instance(p, 0, *a)


@pytest.mark.parametrize("n,m", DIMS)
def test_solve_tvlqr_is_certified(api, n, m):
    """The public path (one instance, boxes indexed by timestep as the reference passes them)."""
    T = 12
    p = bk.make_problem(n, m, T, "tv", "nonsym", I=1, seed=77 + n)
    xb = np.stack((p["xlo"], p["xhi"]))
    # solve_tvlqr also boxes x_0 (an x0 outside row 0 is an infeasible QP, tv_lqr.py:113-114); the generator's
    # box is made for x_1..x_T, so row 0 is opened.  The QP over x_1..x_T does not change.
    xb[0, 0], xb[1, 0] = -bk.BIG, bk.BIG
    ub = np.stack((p["ulo"], p["uhi"]))
    xs, us = api.m.solve_tvlqr(p["At"][0], p["Bt"][0], p["ct"][0], p["Q"], p["Qd"], p["R"], p["x0"][0], p["xd"][0],
                               None, x_bound_abs=xb, u_bound_abs=ub)
    c = bk.instance_qp(p, 0).certify(us)
    assert c["certified"]
    assert np.max(np.abs(us - c["u"])) <= BAR * max(1.0, np.max(np.abs(c["u"])))
    assert np.max(np.abs(xs - c["x"])) <= BAR * max(1.0, np.max(np.abs(c["x"])))


# ------------------------------------------------------------------------------------------------
# MPC mode (mpc = 1): the reference's closed loop on the true dynamics
# ------------------------------------------------------------------------------------------------
def central_difference_tv_matrices(orc, x_trj, u_trj, h=1e-6):
    """An affine model of a system without Jacobians (the three carts' contact resolution): central differences
    of the oracle's dynamics.  Any affine model serves here: the tests are about the QP built on it."""
    T, n, m = u_trj.shape[0], x_trj.shape[1], u_trj.shape[1]
    At, Bt, ct = np.zeros((T, n, n)), np.zeros((T, n, m)), np.zeros((T, n))
    for t in range(T):
        for j in range(n + m):
            d = np.zeros(n + m)
            d[j] = h
            fp = orc.dynamics(x_trj[t] + d[:n], u_trj[t] + d[n:])
            fm = orc.dynamics(x_trj[t] - d[:n], u_trj[t] - d[n:])
            (At[t][:, j] if j < n else Bt[t][:, j - n])[:] = (fp - fm) / (2 * h)
        ct[t] = cr.affine_offset(orc, At[t], Bt[t], x_trj[t], u_trj[t])
    return At, Bt, ct


def mpc_problem(api, mlp, name, T, I):
    """Linearization of the example config around its initial rollout, I start states, an input box that
    the unconstrained closed loop leaves at some start times only."""
    if name == "mlp":
        cfg, system, orc = ec.pendulum_nn(T=T), mlp[0], mlp[1]
    else:
        cfg = ec.CONFIGS[name](T=T)
        system = {"pendulum": api.m.PendulumDynamics, "bicycle": api.m.BicycleDynamics,
                  "quadrotor": api.m.QuadrotorDynamics, "three_cart": api.m.ThreeCartDynamics}[name](cfg["h"])
        orc = {"pendulum": cr.PendulumOracle, "bicycle": cr.BicycleOracle, "quadrotor": cr.QuadrotorOracle,
               "three_cart": cr.ThreeCartOracle}[name](cfg["h"])
    u_init = cfg["u_trj_initial"][:T]
    x_init = cr.rollout(orc, cfg["x0"], u_init)
    if hasattr(orc, "jacobian_xu"):
        At, Bt, ct = cr.exact_tv_matrices(orc, x_init, u_init)
    else:
        At, Bt, ct = central_difference_tv_matrices(orc, x_init, u_init)
    n, m = At.shape[1], Bt.shape[2]
    xd = cfg["xd_trj"][:T + 1]
    K0, k0 = cr.tvlqr_riccati(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], xd)
    rng = np.random.default_rng(T)
    x0 = cfg["x0"] + 0.05 * np.arange(I)[:, None] * rng.standard_normal((I, n))
    u_free = np.concatenate([cr.closed_loop_descent(orc, K0, k0, x0[i])[1] for i in range(I)])
    uc = np.median(u_free, axis=0)
    ua = np.quantile(np.abs(u_free - uc), 0.8, axis=0)
    p = dict(At=np.tile(At, (I, 1, 1, 1)), Bt=np.tile(Bt, (I, 1, 1, 1)), ct=np.tile(ct, (I, 1, 1)), xd=xd[None],
             x0=x0, Q=cfg["Q"], Qd=cfg["Qd"], R=cfg["R"], xlo=np.full(n, -bk.BIG), xhi=np.full(n, bk.BIG),
             ulo=uc - ua, uhi=uc + ua, n=n, m=m, T=T, I=I, shared_xd=True)
    gains = (np.tile(K0, (I, 1, 1, 1)), np.tile(k0, (I, 1, 1)))
    return p, system, orc, gains


MPC_CASES = [(s, T, I) for s in ("pendulum", "bicycle", "three_cart", "mlp") for T, I in ((12, 1), (40, 3))]
# the quadrotor at T = 12 tracks its helix with inputs of +-80: the ADMM needs ~5e4 iterations per QP there, and
# a perturbed start does not converge in 1e5, so the several-instance run is at T = 40
MPC_CASES += [("quadrotor", 12, 1), ("quadrotor", 40, 3)]
MPC_CASES.append(("quadrotor", 65, 1))


@pytest.mark.parametrize("name,T,I", MPC_CASES)
def test_mpc_applies_the_certified_first_input(api, mlp, name, T, I):
    p, system, orc, gains = mpc_problem(api, mlp, name, T, I)
    n, m = p["n"], p["m"]
    xa, ua, ca, sa, ita = solve(api, p, mpc=True, system=system)
    xb, ub, cb, sb, itb = solve(api, p, mpc=True, system=system, gains=gains)
    assert np.all(sa == 0) and np.all(sb == 0)
    assert np.all(ita > 0)
    dyn_tol = 1e-5 if name == "mlp" else 1e-12               # the network runs in float32
    n_active = 0
    for i in range(I):
        # the true dynamics
        for x, u in ((xa[i], ua[i]), (xb[i], ub[i])):
            assert np.array_equal(x[0], p["x0"][i])
            for t in range(T):
                f = orc.dynamics(x[t], u[t])
                assert np.max(np.abs(x[t + 1] - f)) <= dyn_tol * max(1.0, np.max(np.abs(f))), (i, t)
        # with and without the skip path: the same first minimiser.  Later on the closed loop amplifies
        # differences below the bar (open-loop unstable systems, changes of the active set)
        assert np.max(np.abs(ub[i][0] - ua[i][0])) <= BAR * max(1.0, np.max(np.abs(ua[i][0]))), i
        for x, u, c_ in ((xa[i], ua[i], ca[i]), (xb[i], ub[i], cb[i])):
            assert abs(c_ - cr.evaluate_cost(x, u, p["xd"][0], p["Q"], p["R"])) <= 1e-12 * abs(c_)
        # every applied input of the run with the skip path (what local_descent runs) is the first input of
        # the QP from the actual state over [t0, T): the candidate plan comes from a single-QP solve, the
        # certificate decides
        for x, u in ((xb[i], ub[i]),):
            for t0 in range(T):
                sub = dict(p, T=T - t0, I=1, At=p["At"][i:i + 1, t0:], Bt=p["Bt"][i:i + 1, t0:],
                           ct=p["ct"][i:i + 1, t0:], xd=p["xd"][:, t0:], x0=x[t0][None])
                _, us, _, st, _ = solve(api, sub)
                assert st[0] == 0
                c = bk.instance_qp(sub, 0).certify(us[0])
                assert c["certified"], (i, t0)
                n_active += int(np.any(c["active"]))
                assert np.max(np.abs(u[t0] - c["u"][0])) <= BAR * max(1.0, np.max(np.abs(c["u"]))), (i, t0)
    assert n_active > 0
    if T <= 12:
        for i in range(I):
            xo, uo, _ = bq.mpc_box_descent(orc, p["At"][i], p["Bt"][i], p["ct"][i], p["Q"], p["Qd"], p["R"], p["x0"][i],
                                           p["xd"][0], p["xlo"], p["xhi"], p["ulo"], p["uhi"],
                                           gains0=(gains[0][i], gains[1][i]))
            assert np.max(np.abs(ub[i][0] - uo[0])) <= BAR * max(1.0, np.max(np.abs(uo[0])))
            assert np.max(np.abs(ub[i] - uo)) <= 1e-5 * max(1.0, np.max(np.abs(uo)))
            assert np.max(np.abs(xb[i] - xo)) <= 1e-5 * max(1.0, np.max(np.abs(xo)))


# ------------------------------------------------------------------------------------------------
# failure flags
# ------------------------------------------------------------------------------------------------
def test_max_iter_one_flags_only_instances_that_run_the_admm(api):
    """MPC with the skip path and max_iter = 1: an instance whose unconstrained plans all stay inside the box
    runs no ADMM and succeeds; the others fail.  Pendulum, input box +-2: the plans from (2.5, 0.5) reach
    |u| = 1.34 at most, those from (0, 0) and (-0.5, 0) pass 2 in their first plan."""
    T, I = 12, 3
    p, system, orc, gains = mpc_problem(api, None, "pendulum", T, I)
    p["x0"] = np.array([[0.0, 0.0], [2.5, 0.5], [-0.5, 0.0]])
    p["ulo"], p["uhi"] = np.array([-2.0]), np.array([2.0])
    _, _, _, st, it = solve(api, p, mpc=True, system=system, gains=gains, max_iter=1)
    assert it[1] == 0 and st[1] == 0
    assert np.all(st[[0, 2]] == 1) and np.all(it[[0, 2]] > 0)
    _, _, _, st, _ = solve(api, p, mpc=True, system=system, gains=gains)
    assert np.all(st == 0)


def test_nan_flags_exactly_that_instance(api):
    T, I = 12, 3
    p = bk.make_problem(5, 2, T, "both", "dense", I=I, seed=3)
    x, u, cost, status, iters = solve(api, p)
    assert np.all(status == 0)
    p["ct"] = p["ct"].copy()
    p["ct"][1, 4, 0] = np.nan
    _, _, _, st, _ = solve(api, p, max_iter=10 * int(iters.max()))
    assert np.array_equal(st, np.array([0, 1, 0], np.int32))


def test_unreachable_state_box_fails(api, monkeypatch):
    """x_1 boxed far beyond what the boxed input can reach: status 1 after max_iter, and solve_tvlqr raises."""
    n, m, T = 5, 2, 6
    p = bk.make_problem(n, m, T, "input", "diag", I=1, seed=11)
    xlo, xhi = np.full((T + 1, n), -1e4), np.full((T + 1, n), 1e4)
    xlo[1, 0] = 1e3
    p["xlo"], p["xhi"] = xlo, xhi
    _, _, _, st, it = solve(api, p, max_iter=500)
    assert st[0] == 1 and it[0] == 500
    monkeypatch.setattr(api.tv, "box_solve_device", functools.partial(api.tv.box_solve_device, max_iter=500))
    with pytest.raises(ValueError, match="TV_LQR failed"):
        api.m.solve_tvlqr(p["At"][0], p["Bt"][0], p["ct"][0], p["Q"], p["Qd"], p["R"], p["x0"][0], p["xd"][0], None,
                          x_bound_abs=np.stack((xlo, xhi)),
                          u_bound_abs=np.stack((np.tile(p["ulo"], (T, 1)), np.tile(p["uhi"], (T, 1)))))
