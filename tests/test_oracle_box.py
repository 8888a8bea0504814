"""CPU checks of the box-constrained TVLQR oracle (oracle/box_tvlqr.py): the ADMM restatement of the
reference's bounded QP (irs_lqr/tv_lqr.py:69-137 with :113-118,:132-134) against an independent dense
QP solve, its independence from the penalty parameter, and the MPC loop of irs_lqr.py:169-184."""
import numpy as np
import pytest

from oracle import box_kkt as bk
from oracle import box_tvlqr as bq
from oracle import cpu_restatement as cr
from oracle import example_configs as ec


def _problem(T, u_const=(0.5, 0.6)):
    cfg = ec.bicycle(T=T)
    orc = cr.BicycleOracle(cfg["h"])
    u0 = np.tile(np.array(u_const), (T, 1))
    x_trj = cr.rollout(orc, cfg["x0"], u0)
    At, Bt, ct = cr.exact_tv_matrices(orc, x_trj, u0)
    return cfg, orc, At, Bt, ct


def test_admm_matches_dense_qp_and_respects_bounds():
    T = 10
    cfg, orc, At, Bt, ct = _problem(T)
    xlo, xhi = np.array([-1e4, -1e4, -1e4, -1e4, -0.3]), np.array([1e4, 1e4, 1e4, 1e4, 0.3])
    ulo, uhi = np.array([-1e4, -0.4]), np.array([1e4, 0.4])
    x, u, it = bq.admm_box_qp(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], xlo, xhi, ulo, uhi)
    xr, ur, res = bq.dense_qp_reference(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], xlo, xhi,
                                        ulo, uhi)
    assert res.success and it < bq.DEFAULT_MAX_ITER
    np.testing.assert_allclose(u, ur, rtol=0, atol=2e-5)
    np.testing.assert_allclose(x, xr, rtol=0, atol=2e-5)
    assert np.max(np.abs(x[1:, 4])) <= 0.3 + 1e-6 and np.max(np.abs(u[:, 1])) <= 0.4 + 1e-6
    assert np.max(np.abs(x[:, 4])) > 0.29


def test_inactive_bounds_reduce_to_the_riccati_solution():
    T = 15
    cfg, orc, At, Bt, ct = _problem(T, (0.1, 0.0))
    big = 1e6
    x, u, _ = bq.admm_box_qp(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], -big * np.ones(5),
                             big * np.ones(5), -big * np.ones(2), big * np.ones(2))
    xs, us = cr.solve_tvlqr(At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"])
    np.testing.assert_allclose(u, us, rtol=0, atol=1e-7)
    np.testing.assert_allclose(x, xs, rtol=0, atol=1e-7)


@pytest.mark.parametrize("rho0", [0.2, 5.0])
def test_mpc_descent_is_independent_of_the_penalty(rho0):
    """The closed-loop result is the sequence of QP minimisers, not an artefact of the ADMM penalty."""
    T = 20
    cfg = ec.bicycle(T=T)
    orc = cr.BicycleOracle(cfg["h"])
    x_trj = cr.rollout(orc, cfg["x0"], cfg["u_trj_initial"])
    At, Bt, ct = cr.exact_tv_matrices(orc, x_trj, cfg["u_trj_initial"])
    args = (orc, At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"], cfg["xbound"][0],
            cfg["xbound"][1], cfg["ubound"][0], cfg["ubound"][1])
    x1, u1, _ = bq.mpc_box_descent(*args)
    x2, u2, _ = bq.mpc_box_descent(*args, rho0=rho0)
    np.testing.assert_allclose(u1, u2, rtol=0, atol=1e-7)
    np.testing.assert_allclose(x1, x2, rtol=0, atol=1e-7)
    assert np.max(np.abs(x1[:, 4])) <= np.pi / 4 + 1e-6
    assert cr.evaluate_cost(x1, u1, cfg["xd_trj"], cfg["Q"], cfg["R"]) < \
        cr.evaluate_cost(x_trj, cfg["u_trj_initial"], cfg["xd_trj"], cfg["Q"], cfg["R"])


# ------------------------------------------------------------------------------------------------
# the KKT certificate (oracle/box_kkt.py) and the ADMM's accuracy against it
# ------------------------------------------------------------------------------------------------
BAR = 1e-7          # max |u - u*|, max |x - x*| <= BAR max(1, |.*|_inf)


def _steer_problem(T=12):
    """The bicycle with the steer box active (as in the GPU test of solve_tvlqr)."""
    cfg, orc, At, Bt, ct = _problem(T)
    xlo, xhi = np.array([-1e4, -1e4, -1e4, -1e4, -0.3]), np.array([1e4, 1e4, 1e4, 1e4, 0.3])
    ulo, uhi = np.array([-1e4, -0.4]), np.array([1e4, 0.4])
    return (At, Bt, ct, cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"], cfg["xd_trj"]), (xlo, xhi, ulo, uhi)


def _generated(n, m, T, box, kind, i=0):
    p = bk.make_problem(n, m, T, box, kind, I=2, seed=17 * n + T)
    args = (p["At"][i], p["Bt"][i], p["ct"][i], p["Q"], p["Qd"], p["R"], p["x0"][i], p["xd"][i])
    return args, (p["xlo"], p["xhi"], p["ulo"], p["uhi"])


def _within_bar(a, ref):
    return float(np.max(np.abs(a - ref))) <= BAR * max(1.0, float(np.max(np.abs(ref))))


CASES = [("steer", None, None, None, None)] + [
    ("gen", n, m, box, kind) for n, m in ((2, 1), (5, 2), (6, 2), (12, 4)) for box, kind in
    (("input", "dense"), ("state", "diag"), ("both", "nonsym"), ("tv", "dense"))]


def _case(c, T=12):
    return _steer_problem(T) if c[0] == "steer" else _generated(c[1], c[2], T, c[3], c[4])


@pytest.mark.parametrize("case", CASES, ids=lambda c: "-".join(str(v) for v in c if v is not None))
def test_admm_meets_the_accuracy_bar_against_the_certificate(case):
    args, box = _case(case)
    x, u, it = bq.admm_box_qp(*args, *box)
    qp = bk.BoxQP(*args, *box)
    c = qp.certify(u)
    assert c["certified"], (c["min_lam"], c["max_violation"], c["kkt_residual"])
    assert np.any(c["active"])
    lam_rel, slack_rel = qp.margins(c)
    assert lam_rel >= 1e-8 and slack_rel >= 1e-5           # strictly complementary: the active set is unambiguous
    assert _within_bar(u, c["u"]) and _within_bar(x, c["x"]), (np.max(np.abs(u - c["u"])), np.max(np.abs(x - c["x"])))


@pytest.mark.parametrize("case", CASES[:5], ids=lambda c: "-".join(str(v) for v in c if v is not None))
def test_certificate_agrees_with_slsqp(case):
    args, box = _case(case, T=8)
    qp = bk.BoxQP(*args, *box)
    xr, ur, res = bq.dense_qp_reference(*args, *box)
    assert res.success
    c = qp.certify(ur, delta=1e-5)
    assert c["certified"]
    # SLSQP stops at its own floor (~1e-8); the certificate is exact
    np.testing.assert_allclose(ur, c["u"], rtol=0, atol=1e-6 * max(1.0, np.max(np.abs(c["u"]))))
    np.testing.assert_allclose(xr, c["x"], rtol=0, atol=1e-6 * max(1.0, np.max(np.abs(c["x"]))))


@pytest.mark.parametrize("n,m,kind", [(2, 1, "diag"), (5, 2, "dense"), (6, 2, "nonsym"), (12, 4, "dense")])
def test_certificate_agrees_with_bvls_on_input_boxes(n, m, kind):
    p = bk.make_problem(n, m, 30, "input", kind, I=1, seed=n + m)
    qp = bk.instance_qp(p, 0)
    ub, res = bk.bvls(qp, p["Q"], p["Qd"], p["R"], p["ulo"], p["uhi"])
    assert res.status > 0
    c = qp.certify(ub)
    assert c["certified"] and np.sum(c["active"]) >= 2
    assert float(np.max(np.abs(ub - c["u"]))) <= 1e-9 * max(1.0, float(np.max(np.abs(c["u"]))))


def test_certificate_rejects_a_perturbed_or_incomplete_candidate():
    args, box = _steer_problem()
    qp = bk.BoxQP(*args, *box)
    x, u, _ = bq.admm_box_qp(*args, *box)
    c = qp.certify(u)
    assert c["certified"] and np.sum(c["active"]) >= 2
    # a candidate 1e-6 away from the minimiser: the certificate's point is the minimiser, not the candidate
    bad = c["u"] + 1e-6 * np.sign(np.random.default_rng(0).standard_normal(c["u"].shape))
    cb = qp.certify(bad)
    assert cb["certified"] and np.array_equal(cb["active"], c["active"])
    assert not _within_bar(bad, cb["u"])
    # an active set with one constraint dropped: that row is violated at the resulting point
    for row in np.flatnonzero(c["active"]):
        act = c["active"].copy()
        act[row] = False
        r = qp.at(act)
        assert not r["certified"] and r["max_violation"] > 1e-6, row
    # and one with a spurious row added: its multiplier is negative
    extra = c["active"].copy()
    extra[int(np.argmin(np.where(c["active"], np.inf, qp.slack(c["u"]))))] = True
    assert not qp.at(extra)["certified"]


@pytest.mark.parametrize("case", CASES[:5], ids=lambda c: "-".join(str(v) for v in c if v is not None))
def test_admm_is_invariant_under_a_scaling_of_the_weights(case):
    """The QP and its minimiser do not change when (Q, Qd, R) are scaled together, and neither may the solve:
    bit-identical at 2^+-100 (every step is homogeneous and powers of two are exact), 1e-12 at 1e+-30.  Each
    scaled solve gets ten times the iterations of the unscaled one."""
    args, box = _case(case)
    At, Bt, ct, Q, Qd, R, x0, xd = args
    x, u, it = bq.admm_box_qp(*args, *box)
    for s in (2.0 ** 100, 2.0 ** -100, 1e30, 1e-30):
        xs, us, its = bq.admm_box_qp(At, Bt, ct, s * Q, s * Qd, s * R, x0, xd, *box, max_iter=10 * it)
        if s in (2.0 ** 100, 2.0 ** -100):
            assert its == it and np.array_equal(us, u) and np.array_equal(xs, x), s
        else:
            assert np.max(np.abs(us - u)) <= 1e-12 * max(1.0, np.max(np.abs(u))), s
            assert np.max(np.abs(xs - x)) <= 1e-12 * max(1.0, np.max(np.abs(x))), s
