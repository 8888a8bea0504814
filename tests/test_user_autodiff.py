"""User-written dynamics differentiated on the device: CudaSourceDynamics(..., autodiff=True) (GPU tests: -m gpu).

With autodiff the library evaluates the step body over forward-mode dual numbers (csrc/dual.cuh) and reads the
Jacobian off the tangents, so first order, exact and the Jacobian methods need no hand-written Jacobian body.

Test systems:
- the bodies of test_user_dynamics.py (pendulum, bicycle, cart-pole, the (6, 3) drag system), whose hand-written
  Jacobians or float64 oracles are the reference;
- oracle/user_grid.py's body at pairs that take one pass, exactly one full pass, and two passes with a short
  last block of tangent lanes;
- the quadrotor written as source (the double expression form of csrc/systems.cuh), against the built-in
  system's generated Jacobian;
- a calculus system whose step uses every supported operation and a branchy system (branches on values, fabs,
  fmin / fmax, saturation), each with a float64 numpy twin differentiated by complex step.
"""
import concurrent.futures
import ctypes
import json
import os

import numpy as np
import pytest

import test_user_dynamics as tud
from irs_mpc_b200 import _lib, user_system
from oracle import cpu_restatement as cr
from oracle import example_configs as ec
from oracle import sample_gram as sg
from oracle import user_grid as ug

QUADROTOR_STEP = """
    const auto mass = p[0], L = p[1], g = p[2], I0 = p[3], I1 = p[4], I2 = p[5], kF = p[6], kM = p[7];
    R sr, cr, sp, cp, sy, cy;
    Math<R>::sincos(x[3], sr, cr);
    Math<R>::sincos(x[4], sp, cp);
    Math<R>::sincos(x[5], sy, cy);
    const R icp = Math<R>::rcp(cp);
    const R rd0 = x[9], rd1 = x[10], rd2 = x[11];
    const R s03 = u[0] + u[3], s12 = u[1] + u[2];
    const R Fz = kF * (s03 + s12);
    const R M0 = (L * kF) * ((u[2] + u[3]) - (u[0] + u[1]));
    const R M1 = (L * kF) * (s12 - s03);
    const R M2 = kM * ((u[1] + u[3]) - (u[0] + u[2]));
    const R a = Fz * (1 / mass);
    const R spcr = sp * cr;
    o[6] = x[6] + h * (a * (cy * spcr + sy * sr));
    o[7] = x[7] + h * (a * (sy * spcr - cy * sr));
    o[8] = x[8] + h * (a * (cp * cr) - g);
    const R cprd2 = cp * rd2;
    const R pr = rd0 - sp * rd2;
    const R q = cr * rd1 + sr * cprd2;
    const R r = cr * cprd2 - sr * rd1;
    const R pd = (M0 + (I1 - I2) * (q * r)) * (1 / I0);
    const R qd = (M1 + (I2 - I0) * (r * pr)) * (1 / I1);
    const R rdd = (M2 + (I0 - I1) * (pr * q)) * (1 / I2);
    const R tp = sp * icp;
    const R icp2 = icp * icp;
    const R srq_crr = sr * q + cr * r;
    const R crq_srr = cr * q - sr * r;
    const R srqd_crrd = sr * qd + cr * rdd;
    o[9] = x[9] + h * (pd + tp * srqd_crrd + rd0 * (tp * crq_srr) + rd1 * (icp2 * srq_crr));
    o[10] = x[10] + h * ((cr * qd - sr * rdd) - rd0 * srq_crr);
    o[11] = x[11] + h * (icp * srqd_crrd + rd0 * (icp * crq_srr) + rd1 * (tp * icp * srq_crr));
    for (int i = 0; i < 6; ++i) o[i] = x[i] + h * x[6 + i];
"""
QUADROTOR_PARAMS = [0.775, 0.15, 9.81, 0.0015, 0.0025, 0.0035, 1.0, 0.0245]      # systems.py: QuadrotorDynamics

# every supported operation; (5, 4): two passes of five lanes
CALCULUS_STEP = """
    const R a0 = R(1.5) + sin(x[0]);
    const R sq = sqrt(R(1) + x[1] * x[1]);
    const R ex = exp(R(-0.5) * x[2]);
    const R lg = log(2 + cos(x[3]));
    const R tn = tan(0.3f * x[4]);
    const R as = asin(R(0.5) * tanh(u[0]));
    const R ac = acos(0.4 * sin(u[1]));
    const R at = atan(x[0] * u[2]);
    const R a2 = atan2(x[1] + R(0.2), R(1.5) + cos(u[3]));
    using B = decltype(h);                      // float / double: the plain atan2 / fmin / fmax want one type
    const R a3 = atan2(x[2], B(2)) + atan2(B(1), R(2) + x[3] * x[3]);
    const R hy = sinh(R(0.5) * u[0]) * cosh(R(0.5) * u[1]);
    const R pw = pow(a0, 1.5) + pow(sq, 2);
    const R ab = fabs(x[2] - u[3]);
    const R mn = fmin(x[3], u[0]) + fmin(x[4], B(0.25)) + fmin(B(-0.25), u[1]);
    const R mx = fmax(x[4], R(0.5) * u[1]) + fmax(x[0], B(-0.3)) + fmax(B(0.3), u[2]);
    R s, c;
    Math<R>::sincos(x[4], s, c);
    const R rc = Math<R>::rcp(R(2) + c);
    const R dv = Math<R>::div(x[0], R(3) + s);
    R acc = x[0];
    acc += sq * h;
    acc -= 0.1 * ex;
    acc *= R(1) + R(0.01) * lg;
    acc /= R(1.2) + 0.1 * s;
    R t = -tn;
    t += 1;
    t -= 0.5f;
    t *= 2;
    t /= 3;
    o[0] = acc + h * (as * ac - at / (1 + a2 * a2));
    o[1] = x[1] + h * (hy - pw / 4 + ab);
    o[2] = x[2] + h * (mn * mx + rc - dv * t);
    o[3] = 1 - x[3] * 0.5 + h * (a3 - 2 / (R(3) + x[1] * x[1]) + (x[0] - 1) * u[3]);
    o[4] = (x[4] + h * (u[0] * u[1] - u[2] * u[3])) / 1.5 + x[0] / R(4);
    if (x[0] > 0.0 && 0.0 < x[1] && x[2] >= R(-10) && R(10) <= 100 + x[3] && x[4] != 7 && x[4] <= 7.0 &&
        !(x[0] == R(-7)) && x[0] < 7)
        o[4] += h * x[2];
"""

# branches on values, fabs, fmin / fmax and saturation; (3, 2)
BRANCHY_STEP = """
    R v = x[1] + h * u[0];
    if (v > R(1)) v = R(1) + R(0.1) * (v - R(1));
    else if (v < R(-1)) v = R(-1) + R(0.1) * (v + R(1));
    const R sat = fmin(fmax(u[1], R(-0.5)), R(0.5));
    o[0] = x[0] + h * v;
    o[1] = v - h * fmin(x[0], x[2]);
    o[2] = x[2] + h * (sat + fabs(x[0]) * x[2]) + h * fmax(x[1] * x[2], u[0]);
    if (x[0] * u[1] > R(0)) o[2] += h * x[0] * u[1];
"""
CALC_H, BRANCHY_H = 0.1, 0.1

GRID_AD = [(1, 1), (7, 1), (8, 1), (4, 7), (10, 3), (8, 8), (12, 4)]
GRID_IDS = ["%dx%d" % nm for nm in GRID_AD]

# name -> (dim_x, dim_u, h, params, step); every one built with autodiff=True
AD_SPECS = {
    "pendulum_ad": (2, 1, 0.05, [], tud.PENDULUM_STEP),
    "bicycle_ad": (5, 2, 0.1, [], tud.BICYCLE_STEP),
    "cartpole_ad": (4, 1, 0.02, tud.CARTPOLE_PARAMS, tud.CARTPOLE_STEP),
    "drag3d_ad": (6, 3, 0.05, [0.2], tud.DRAG_STEP),
    "quadrotor_ad": (12, 4, 0.05, QUADROTOR_PARAMS, QUADROTOR_STEP),
    "calculus_ad": (5, 4, CALC_H, [], CALCULUS_STEP),
    "branchy_ad": (3, 2, BRANCHY_H, [], BRANCHY_STEP),
}
AD_SPECS.update({"grid_ad_%d_%d" % nm: (nm[0], nm[1], ug.H, ug.PARAMS, ug.step_source()) for nm in GRID_AD})
# the same steps without autodiff: hand-written Jacobian bodies, or none
HAND_SPECS = {name: tud.SPECS[name] for name in ("pendulum_src", "bicycle_src", "cartpole", "cartpole_nojac",
                                                 "drag3d")}
HAND_SPECS.update({"grid_%d_%d" % nm: (nm[0], nm[1], ug.H, ug.PARAMS, ug.step_source(), ug.jacobian_source())
                   for nm in GRID_AD})
TWIN_OF = {"pendulum_ad": "pendulum_src", "bicycle_ad": "bicycle_src", "cartpole_ad": "cartpole"}


@pytest.fixture(scope="module")
def built():
    """Every library of this module, compiled in parallel (or found in the user cache) -> name: (path, s, hash)."""
    jobs = [(name, (n, m, 1 + len(prm), step, None, name, True)) for name, (n, m, h, prm, step) in AD_SPECS.items()]
    jobs += [(name, (n, m, 1 + len(prm), step, jac, name)) for name, (n, m, h, prm, step, jac) in HAND_SPECS.items()]
    with concurrent.futures.ThreadPoolExecutor(8) as pool:
        futs = {name: pool.submit(user_system.build_library, *args) for name, args in jobs}
        return {name: f.result() for name, f in futs.items()}


_SYSTEMS = {}


def system(built, name):
    if name not in _SYSTEMS:
        if name in AD_SPECS:
            n, m, h, prm, step = AD_SPECS[name]
            s = user_system.CudaSourceDynamics(n, m, h, prm, step=step, autodiff=True, name=name)
        else:
            n, m, h, prm, step, jac = HAND_SPECS[name]
            s = user_system.CudaSourceDynamics(n, m, h, prm, step=step, jacobian=jac, name=name)
        assert s.library_path == built[name][0]
        _SYSTEMS[name] = s
    return _SYSTEMS[name]


@pytest.fixture(scope="module")
def api():
    import irs_mpc_b200.all as a
    return a


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


# ------------------------------------------------------------------------------------------------
# float64 numpy twins of the calculus and branchy systems, differentiated by complex step: branches and
# selections follow the real parts, as the dual numbers follow the values
# ------------------------------------------------------------------------------------------------
def _where(cond, a, b):
    return np.where(cond, a, b)


def _fabs(a):
    return _where(a.real >= 0, a, -a)


def _fmin(a, b):
    a, b = np.broadcast_arrays(a + 0j, b + 0j)
    return _where(b.real < a.real, b, a)


def _fmax(a, b):
    a, b = np.broadcast_arrays(a + 0j, b + 0j)
    return _where(b.real > a.real, b, a)


def _atan2(y, x):
    """atan2 that complex step differentiates: arctan(y / x) plus the quadrant's constant."""
    y, x = np.broadcast_arrays(y + 0j, x + 0j)
    off = np.where(x.real > 0, 0.0, np.where(y.real >= 0, np.pi, -np.pi))
    return np.arctan(y / x) + off


def calculus_f(x, u, h=CALC_H):
    a0 = 1.5 + np.sin(x[:, 0])
    sq = np.sqrt(1 + x[:, 1] ** 2)
    ex = np.exp(-0.5 * x[:, 2])
    lg = np.log(2 + np.cos(x[:, 3]))
    tn = np.tan(np.float64(np.float32(0.3)) * x[:, 4])
    as_ = np.arcsin(0.5 * np.tanh(u[:, 0]))
    ac = np.arccos(0.4 * np.sin(u[:, 1]))
    at = np.arctan(x[:, 0] * u[:, 2])
    a2 = _atan2(x[:, 1] + 0.2, 1.5 + np.cos(u[:, 3]))
    a3 = _atan2(x[:, 2], 2.0) + _atan2(1.0, 2 + x[:, 3] ** 2)
    hy = np.sinh(0.5 * u[:, 0]) * np.cosh(0.5 * u[:, 1])
    pw = np.power(a0, 1.5) + np.power(sq, 2)
    ab = _fabs(x[:, 2] - u[:, 3])
    mn = _fmin(x[:, 3], u[:, 0]) + _fmin(x[:, 4], 0.25) + _fmin(-0.25, u[:, 1])
    mx = _fmax(x[:, 4], 0.5 * u[:, 1]) + _fmax(x[:, 0], -0.3) + _fmax(0.3, u[:, 2])
    s, c = np.sin(x[:, 4]), np.cos(x[:, 4])
    rc = 1 / (2 + c)
    dv = x[:, 0] / (3 + s)
    acc = (x[:, 0] + sq * h - 0.1 * ex) * (1 + 0.01 * lg) / (1.2 + 0.1 * s)
    t = (-tn + 1 - 0.5) * 2 / 3
    o0 = acc + h * (as_ * ac - at / (1 + a2 * a2))
    o1 = x[:, 1] + h * (hy - pw / 4 + ab)
    o2 = x[:, 2] + h * (mn * mx + rc - dv * t)
    o3 = 1 - x[:, 3] * 0.5 + h * (a3 - 2 / (3 + x[:, 1] ** 2) + (x[:, 0] - 1) * u[:, 3])
    o4 = (x[:, 4] + h * (u[:, 0] * u[:, 1] - u[:, 2] * u[:, 3])) / 1.5 + x[:, 0] / 4
    o4 = o4 + _where((x[:, 0].real > 0) & (x[:, 1].real > 0), h * x[:, 2], 0)
    return np.stack([o0, o1, o2, o3, o4], 1)


def branchy_f(x, u, h=BRANCHY_H):
    v = x[:, 1] + h * u[:, 0]
    v = _where(v.real > 1, 1 + 0.1 * (v - 1), _where(v.real < -1, -1 + 0.1 * (v + 1), v))
    sat = _fmin(_fmax(u[:, 1], -0.5), 0.5)
    o0 = x[:, 0] + h * v
    o1 = v - h * _fmin(x[:, 0], x[:, 2])
    o2 = x[:, 2] + h * (sat + _fabs(x[:, 0]) * x[:, 2]) + h * _fmax(x[:, 1] * x[:, 2], u[:, 0])
    o2 = o2 + _where((x[:, 0] * u[:, 1]).real > 0, h * x[:, 0] * u[:, 1], 0)
    return np.stack([o0, o1, o2], 1)


def branchy_margins(x, u, h=BRANCHY_H):
    """Distance of each point to every kink of the branchy step -> [points, kinks] (and the sides: sign)."""
    v = x[:, 1] + h * u[:, 0]
    return np.stack([v - 1, v + 1, u[:, 1] + 0.5, u[:, 1] - 0.5, x[:, 0], x[:, 0] - x[:, 2],
                     x[:, 1] * x[:, 2] - u[:, 0], u[:, 1]], 1)


def complex_step_jacobian(f, x, u):
    n, m = x.shape[1], u.shape[1]
    xu = np.hstack((x, u)).astype(np.complex128)
    eps = 1e-30
    J = np.zeros((xu.shape[0], n, n + m))
    for j in range(n + m):
        z = xu.copy()
        z[:, j] += 1j * eps
        J[:, :, j] = f(z[:, :n], z[:, n:]).imag / eps
    return J


class TwinOracle:
    def __init__(self, f, n, m, h):
        self.f, self.dim_x, self.dim_u, self.h = f, n, m, h

    def dynamics_batch(self, x, u):
        return self.f(np.atleast_2d(x) + 0j, np.atleast_2d(u) + 0j).real

    def jacobian_xu_batch(self, x, u):
        return complex_step_jacobian(self.f, np.atleast_2d(x), np.atleast_2d(u))


class DragJacOracle(tud.DragOracle):
    """test_user_dynamics.DragOracle with its analytic Jacobian."""

    def jacobian_xu_batch(self, x, u):
        x, u = np.atleast_2d(x), np.atleast_2d(u)
        h, c = self.h, self.drag
        v = x[:, 3:]
        sp = np.sqrt(1.0 + np.sum(v ** 2, axis=1))
        I3 = np.eye(3)[None]
        dvv = I3 * (1 - h * c * sp)[:, None, None] - h * c * v[:, :, None] * v[:, None, :] / sp[:, None, None]
        J = np.zeros((x.shape[0], 6, 9))
        J[:, :3, :3] = I3
        J[:, :3, 3:6] = h * dvv
        J[:, :3, 6:] = h * h * I3
        J[:, 3:, 3:6] = dvv
        J[:, 3:, 6:] = h * I3
        return J

    def jacobian_xu(self, x, u):
        return self.jacobian_xu_batch(x, u)[0]


# ------------------------------------------------------------------------------------------------
# CPU: the keyword, the build, the loud failure
# ------------------------------------------------------------------------------------------------
def test_jacobian_and_autodiff_together_are_refused_before_compiling(monkeypatch):
    monkeypatch.setattr(user_system, "_compile", lambda *a: pytest.fail("compiled"))
    with pytest.raises(ValueError, match="not both"):
        user_system.CudaSourceDynamics(2, 1, 0.05, [], step=tud.PENDULUM_STEP, jacobian=tud.PENDULUM_JAC,
                                       autodiff=True)
    with pytest.raises(ValueError, match="not both"):
        user_system.build_library(2, 1, 1, tud.PENDULUM_STEP, tud.PENDULUM_JAC, "both", True)


def test_generated_source_without_autodiff_does_not_see_dual_numbers():
    for jac in (None, tud.CARTPOLE_JAC):
        src = user_system.generate_source(4, 1, 5, tud.CARTPOLE_STEP, jac)
        assert src == user_system.generate_source(4, 1, 5, tud.CARTPOLE_STEP, jac, False)
        assert "dual.cuh" not in src and "IRS_USER_AUTODIFF" not in src
    src = user_system.generate_source(4, 1, 5, tud.CARTPOLE_STEP, None, True)
    assert '#include "dual.cuh"' in src and src.count(tud.CARTPOLE_STEP.strip().splitlines()[0]) == 1


@pytest.mark.parametrize("d,passes,lanes", [(2, 1, 2), (8, 1, 8), (9, 2, 5), (11, 2, 6), (13, 2, 7), (16, 2, 8)])
def test_pass_plan(d, passes, lanes):
    assert user_system.autodiff_passes(d) == (passes, lanes)


@pytest.mark.parametrize("name", sorted(AD_SPECS))
def test_autodiff_library_loads_and_reports_its_system(built, name):
    n, m = AD_SPECS[name][:2]
    lib = _lib.Library.at(built[name][0])
    assert lib.handle().irs_abi_version() == _lib.ABI_VERSION
    dims = [ctypes.c_int() for _ in range(3)]
    lib.call("irs_system_dims", user_system.USER_SYSTEM_ID, *[ctypes.byref(v) for v in dims])
    assert [v.value for v in dims] == [n, m, n * (n + m)]


def test_autodiff_sources_hash_apart(built):
    pairs = [("cartpole_ad", "cartpole_nojac"), ("drag3d_ad", "drag3d"), ("pendulum_ad", "pendulum_src")]
    pairs += [("grid_ad_%d_%d" % nm, "grid_%d_%d" % nm) for nm in GRID_AD]
    for a, b in pairs:
        assert built[a][2] != built[b][2] and built[a][0] != built[b][0], (a, b)


def test_dropping_the_derivative_does_not_compile(tmp_path, monkeypatch):
    monkeypatch.setenv("IRS_USER_CACHE", str(tmp_path))
    body = "R s, c;\nMath<R>::sincos(x[0], s, c);\nfloat t = x[1];\no[1] = x[1] + h * (u[0] - s) + R(0) * t;\no[0] = x[0];\n"
    # the plain step compiles: the derivative is what is dropped
    user_system.generate_source(2, 1, 1, body)
    with pytest.raises(RuntimeError, match=r"step\(3\)"):
        user_system.build_library(2, 1, 1, body, None, "drops", True)


# ------------------------------------------------------------------------------------------------
# GPU 1, 2: Jacobians in fp64 exact to rounding, in fp32 no worse than the hand-written bodies
# ------------------------------------------------------------------------------------------------
def points(name, count=4096, seed=5):
    n, m = AD_SPECS[name][:2]
    rng = np.random.default_rng(seed)
    if name == "branchy_ad":
        x, u = 1.6 * rng.standard_normal((4 * count, n)), 1.6 * rng.standard_normal((4 * count, m))
        x[:, 1] *= 4.0                                      # v = x1 + h u0 on both sides of +-1
        keep = np.all(np.abs(branchy_margins(x, u)) > 1e-3, axis=1)
        x, u = x[keep][:count], u[keep][:count]
        side = np.sign(branchy_margins(x, u))
        assert np.all((side > 0).sum(axis=0) >= 50) and np.all((side < 0).sum(axis=0) >= 50)
        return x, u
    scale = 0.5 if name == "quadrotor_ad" else 0.7
    x, u = scale * rng.standard_normal((count, n)), scale * rng.standard_normal((count, m))
    if name == "quadrotor_ad":
        u += 2.0                                            # rotor commands near hover
    return x, u


def truth(built, api, name, x, u):
    """The float64 Jacobian the autodiff one is compared with, and the fp32 Jacobian of a hand-written (or
    built-in) body at the same points (None where there is none)."""
    import torch
    n, m = AD_SPECS[name][:2]
    if name in TWIN_OF:
        hand = system(built, TWIN_OF[name])
        return hand.jacobian_xu_batch(x, u), hand.jacobian_xu_batch(x, u, dtype=torch.float32)
    if name.startswith("grid_ad_"):
        hand = system(built, name.replace("grid_ad_", "grid_"))
        return ug.GridOracle(n, m).jacobian_xu_batch(x, u), hand.jacobian_xu_batch(x, u, dtype=torch.float32)
    if name == "quadrotor_ad":
        q = api.QuadrotorDynamics(AD_SPECS[name][2])
        return q.jacobian_xu_batch(x, u), q.jacobian_xu_batch(x, u, dtype=torch.float32)
    if name == "drag3d_ad":
        return DragJacOracle(0.05).jacobian_xu_batch(x, u), None
    f = {"calculus_ad": calculus_f, "branchy_ad": branchy_f}.get(name)
    if f is not None:
        return complex_step_jacobian(f, x, u), None
    return None, None


FP64_CASES = ["pendulum_ad", "bicycle_ad", "cartpole_ad", "drag3d_ad", "quadrotor_ad", "calculus_ad", "branchy_ad"]
FP64_CASES += ["grid_ad_%d_%d" % nm for nm in GRID_AD]


@pytest.mark.gpu
@pytest.mark.parametrize("name", FP64_CASES)
def test_fp64_jacobian_exact_to_rounding(built, api, name):
    s = system(built, name)
    x, u = points(name)
    # at float32-representable points, so that the fp32 comparison below sees the very same inputs
    x, u = x.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)
    J = s.jacobian_xu_batch(x, u)
    ref, hand32 = truth(built, api, name, x, u)
    assert np.all(np.isfinite(J))
    scale = max(1.0, float(np.abs(ref).max()))
    err = float(np.abs(J - ref).max())
    assert err <= 1e-12 * scale, (name, err, scale)
    if name in ("calculus_ad", "branchy_ad"):
        np.testing.assert_allclose(s.dynamics_batch(x, u), TwinOracle(
            calculus_f if name == "calculus_ad" else branchy_f, *AD_SPECS[name][:3]).dynamics_batch(x, u),
            rtol=0, atol=1e-13)
    if hand32 is not None:
        import torch
        J32 = s.jacobian_xu_batch(x, u, dtype=torch.float32).astype(np.float64)
        e_ad = float(np.abs(J32 - ref).max())
        e_hand = float(np.abs(hand32.astype(np.float64) - ref).max())
        assert e_ad <= 2.0 * e_hand + 1e-7 * float(np.abs(ref).max()), (name, e_ad, e_hand)


# ------------------------------------------------------------------------------------------------
# GPU 3: first-order means and the exact linearization on the grid
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("nm", GRID_AD, ids=GRID_IDS)
def test_first_order_means(built, nm, chunk_samples):
    """A_t, B_t against the float64 mean of the library's own fp32 (dual-number) Jacobians at the identical
    perturbed points, per entry in units of mean |J| (the bar of test_user_dims_kernels.py)."""
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    n, m = nm
    s = system(built, "grid_ad_%d_%d" % nm)
    P = 3
    rng = np.random.default_rng(7)
    x_nom, u_nom = 0.5 * rng.standard_normal((P, n)), 0.5 * rng.standard_normal((P, m))
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    sig = 0.05 * (1.0 + 0.15 * np.arange(n + m))
    for N in (1, 2, 33, 129, 257, 4097, 8193):
        for anti in (False, True):
            sampler = sampling.GaussianSampling(sig[:n], sig[n:], N, seed=21, antithetic=anti)
            ws = tsk.guarded_workspace(s, smoothing.FIRST_ORDER, P, N, chunk_samples)
            smoothing.accumulate(s, smoothing.FIRST_ORDER, xd, ud, N, ws, sigma=sampler.sigma(2), seed=21, it=2,
                                 flags=sampler.flags())
            At, Bt, ct, status = smoothing.finalize(s, smoothing.FIRST_ORDER, xd, ud, ws, N)
            torch.cuda.synchronize()
            tsk.check_guard(ws)
            assert not bool(torch.isnan(ws.partials).any())
            assert int(status.sum().item()) == 0
            AB = np.concatenate((_device.to_numpy(At), _device.to_numpy(Bt)), axis=2)
            for p in range(P):
                z = sampler.deltas(1, 2, t0=p)[0]
                pts = (np.concatenate((x_nom[p], u_nom[p])).astype(np.float32)[None, :] + z).astype(np.float32)
                J = s.jacobian_xu_batch(pts[:, :n], pts[:, n:], dtype=torch.float32)
                mean, scale = J.mean(axis=0), np.abs(J).mean(axis=0)
                err = np.abs(AB[p] - mean)
                assert np.all(err[scale == 0] == 0), (N, p)
                r = float(np.max(err[scale > 0] / scale[scale > 0]))
                assert r < sg.TOL_CUDA_CORES, (N, p, anti, r)


@pytest.mark.gpu
@pytest.mark.parametrize("nm", GRID_AD, ids=GRID_IDS)
def test_exact_linearize(built, nm):
    from irs_mpc_b200 import _device
    n, m = nm
    s, orc = system(built, "grid_ad_%d_%d" % nm), ug.GridOracle(n, m)
    P = 77
    rng = np.random.default_rng(4)
    x_nom, u_nom = 0.5 * rng.standard_normal((P, n)), 0.5 * rng.standard_normal((P, m))
    At, Bt, ct = _device.empty((P, n, n)), _device.empty((P, n, m)), _device.empty((P, n))
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    prm, nprm = s._params()
    s.lib.call("irs_exact_linearize", s.system_id, prm, nprm, _device.ptr(xd), _device.ptr(ud), P, _device.ptr(At),
               _device.ptr(Bt), _device.ptr(ct), _device.stream_ptr())
    At_o, Bt_o, ct_o = cr.exact_tv_matrices(orc, x_nom, u_nom)
    assert rel(_device.to_numpy(At), At_o) <= 1e-12 and rel(_device.to_numpy(Bt), Bt_o) <= 1e-12
    assert rel(_device.to_numpy(ct), ct_o) <= 1e-12


# ------------------------------------------------------------------------------------------------
# GPU 4: twins of the hand-Jacobian libraries
# ------------------------------------------------------------------------------------------------
TWIN_CASES = [("pendulum_ad", ec.pendulum), ("bicycle_ad", ec.bicycle), ("cartpole_ad", tud.cartpole_cfg)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfgf", TWIN_CASES)
def test_twin_first_order_and_exact(built, api, name, cfgf):
    T = 30
    cfg = cfgf(T=T)
    s, hand = system(built, name), system(built, TWIN_OF[name])
    n = s.dim_x
    out = []
    for sysm in (s, hand):
        sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], 4000, seed=2)
        solver = api.IrsLqrFirstOrder(sysm, tud.params_of(api, cfg), sampler)
        out.append(solver.get_TV_matrices(solver.x_trj, solver.u_trj))
    for a, b in zip(*out):
        np.testing.assert_allclose(a, b, rtol=0, atol=1e-6 * max(1.0, float(np.abs(b).max())))
    out = []
    for sysm in (s, hand):
        solver = api.IrsLqrExact(sysm, tud.params_of(api, cfg))
        out.append(solver.get_TV_matrices(solver.x_trj, solver.u_trj))
    for a, b in zip(*out):
        assert rel(a, b) <= 1e-12


# ------------------------------------------------------------------------------------------------
# GPU 5: systems without a Jacobian body now run first order and exact
# ------------------------------------------------------------------------------------------------
ORACLE_CASES = [("cartpole_ad", tud.cartpole_cfg, tud.CartPoleOracle), ("drag3d_ad", tud.drag_cfg, DragJacOracle)]


@pytest.mark.gpu
@pytest.mark.parametrize("name,cfgf,oracle", ORACLE_CASES)
def test_first_order_and_exact_against_oracle(built, api, name, cfgf, oracle):
    T, N = 30, 4000
    cfg = cfgf(T)
    s = system(built, name)
    n = s.dim_x
    orc = oracle(cfg["h"])
    sampler = api.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, seed=3)
    solver = api.IrsLqrFirstOrder(s, tud.params_of(api, cfg), sampler)
    At, Bt, ct = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
    deltas = sampler.deltas(T, solver.iter).astype(np.float64)
    At_o, Bt_o, ct_o = cr.first_order_tv_matrices(orc, solver.x_trj, solver.u_trj, deltas)
    assert rel(At, At_o) < 1e-4 and rel(Bt, Bt_o) < 1e-4 and float(np.max(np.abs(ct - ct_o))) < 1e-4
    exact = api.IrsLqrExact(s, tud.params_of(api, cfg))
    At, Bt, ct = exact.get_TV_matrices(exact.x_trj, exact.u_trj)
    At_o, Bt_o, ct_o = cr.exact_tv_matrices(orc, exact.x_trj, exact.u_trj)
    assert rel(At, At_o) < 1e-7 and rel(Bt, Bt_o) < 1e-7
    assert float(np.max(np.abs(ct - ct_o))) < 1e-7 * max(1.0, float(np.abs(ct_o).max()))
    exact.iterate(3, verbose=False)
    assert exact.cost_lst[-1] < exact.cost_lst[0]
    solver.iterate(3, verbose=False)
    assert solver.cost_lst[-1] < solver.cost_lst[0]


# ------------------------------------------------------------------------------------------------
# GPU 6: the step path is untouched
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_order_bit_identical_to_the_plain_build(built, api):
    T = 30
    cfg = tud.cartpole_cfg(T)
    res = []
    for name in ("cartpole_ad", "cartpole_nojac"):
        s = system(built, name)
        sampler = api.GaussianSampling(cfg["sigma"][:4], cfg["sigma"][4:], 3000, seed=5)
        solver = api.IrsLqrZeroOrder(s, tud.params_of(api, cfg), sampler)
        lin = solver.get_TV_matrices(solver.x_trj, solver.u_trj)
        xd, ud = solver.local_descent(solver.x_trj, solver.u_trj)
        x, u, c = solver.iterate(2, verbose=False)
        res.append(lin + (xd, ud, np.array(solver.cost_lst), x, u))
    for i, (a, b) in enumerate(zip(*res)):
        assert np.array_equal(a, b), i


# ------------------------------------------------------------------------------------------------
# GPU 7: the reference's exact loops (pydrake.forwarddiff / symbolic Jacobians) from a step body alone
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("sysname,name,key,rtol", [("pendulum", "pendulum_ad", "pendulum_exact", 1e-10),
                                                   ("quadrotor", "quadrotor_ad", "quadrotor_exact", 1e-7)])
def test_exact_loop_from_source_reproduces_stored_cost_curve(built, api, golden_dir, sysname, name, key, rtol):
    with open(os.path.join(golden_dir, "reference_costs.json")) as f:
        goldc = np.array(json.load(f)["stored_cost_curves"][key]["values"])
    cfg = ec.CONFIGS[sysname]()
    s = system(built, name)
    assert s.h == cfg["h"]
    p = api.IrsLqrParameters()
    p.Q, p.Qd, p.R, p.x0 = cfg["Q"], cfg["Qd"], cfg["R"], cfg["x0"]
    p.xd_trj, p.u_trj_initial = cfg["xd_trj"][:cfg["T"] + 1], cfg["u_trj_initial"][:cfg["T"]]
    p.xbound, p.ubound = cfg["xbound"], cfg["ubound"]
    solver = api.IrsLqrExact(s, p)
    assert abs(solver.cost - goldc[0]) <= 1e-12 * goldc[0]
    solver.iterate(len(goldc) - 2, verbose=False)
    assert len(solver.cost_lst) == len(goldc)
    np.testing.assert_allclose(np.array(solver.cost_lst), goldc, rtol=rtol)
