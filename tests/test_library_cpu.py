"""CPU-side checks: the C-ABI library loads and exports every symbol include/irs_mpc_b200.h
declares, host-only entry points work, and compute entry points fail loudly without a GPU."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "irs_mpc_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(irs_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported_and_bound(built_lib):
    from irs_mpc_b200 import _lib
    names = declared_symbols()
    assert len(names) >= 20
    for name in names:
        assert hasattr(built_lib, name), "library does not export %s" % name
        assert name in _lib.SIGNATURES, "no ctypes signature for %s" % name
    assert sorted(_lib.SIGNATURES) == names
    assert built_lib.irs_abi_version() == _lib.ABI_VERSION == 4


def test_system_dims_and_partial_width(built_lib):
    expect = {0: (2, 1), 1: (5, 2), 2: (12, 4), 3: (6, 2)}
    for sid, (n, m) in expect.items():
        a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert built_lib.irs_system_dims(sid, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)) == 0
        assert (a.value, b.value) == (n, m)
        d = n + m
        # three_cart blocks also carry the first moments [sum z | sum dF] of the centred accumulation
        assert built_lib.irs_partial_width(sid, 0) == d * (d + 1) // 2 + d * n + ((d + n) if sid == 3 else 0)
    assert built_lib.irs_system_dims(9, None, None, None) != 0
    assert b"unknown system" in built_lib.irs_last_error()


@pytest.mark.parametrize("P,N", [(1, 1), (200, 1000), (100, 10000), (100, 100000), (100, 1000000),
                                 (409600, 1000), (3, 77)])
def test_smooth_plan_covers_all_samples(built_lib, P, N):
    from irs_mpc_b200 import smoothing
    for sid in range(4):
        C, S = smoothing.plan(sid, 0, P, N)
        assert C >= 1 and S >= 1 and S % 128 == 0
        assert C * S >= N and (C - 1) * S < N      # no empty chunk
        assert P * C < 2 ** 31


def test_compute_fails_loudly_without_gpu(built_lib):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from irs_mpc_b200 import _lib
    from irs_mpc_b200.all import PendulumDynamics
    with pytest.raises(_lib.IrsCudaError, match="no CPU fallback"):
        PendulumDynamics(0.05).dynamics(np.zeros(2), np.zeros(1))


def test_get_solver_and_sampling_schedule(built_lib):
    from irs_mpc_b200.all import GaussianSampling, get_solver
    assert get_solver("osqp").name == "osqp"
    with pytest.raises(ValueError, match="Do not recognize solver"):
        get_solver("nope")
    s = GaussianSampling([2.0, 4.0], [1.0], 100, power=0.5)
    np.testing.assert_allclose(s.sigma(4), [1.0, 2.0, 0.5])
    assert s.flags() == 8 and s.antithetic                     # antithetic pairs are the default stream
    assert GaussianSampling([2.0, 4.0], [1.0], 100, antithetic=False).flags() == 0
    # the float32 array handed to the kernels is cached per iteration and follows the schedule
    a4, p4 = s.sigma32(4)
    assert a4.dtype == np.float32 and a4.flags["C_CONTIGUOUS"] and s.sigma32(4)[0] is a4
    np.testing.assert_allclose(a4, [1.0, 2.0, 0.5])
    a9, _ = s.sigma32(9)
    assert a9 is not a4
    np.testing.assert_allclose(a9, np.array([2.0, 4.0, 1.0]) / 3.0, rtol=1e-6)
    assert GaussianSampling([1.0], [1.0], 1, projection="absolute").flags() == 2 | 8
    assert GaussianSampling([1.0], [1.0], 1, projection="delta", antithetic=False).flags() == 4
    with pytest.raises(ValueError):
        GaussianSampling([1.0], [1.0], 1, projection="bogus")


def test_drop_in_import_path(built_lib):
    # same import lines as examples/pendulum/pendulum_zero_order.py:8 of the reference
    import subprocess
    import sys
    code = ("from irs_lqr.all import IrsLqrParameters, IrsLqrZeroOrder, IrsLqrFirstOrder, IrsLqrExact;"
            "from irs_lqr.tv_lqr import solve_tvlqr, get_solver;"
            "from irs_lqr.dynamical_system import DynamicalSystem;"
            "p = IrsLqrParameters(); assert p.solver_name == 'osqp'; print('ok')")
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr


def test_argument_validation_messages(built_lib):
    """Host-side validation runs before any launch, so it is testable without a GPU."""
    prm = (ctypes.c_double * 1)(0.05)
    rc = built_lib.irs_smooth_zero_order_accumulate(0, prm, 1, 0, None, None, 1, 10, None, None,
                                                    0, 1, 0, 0, 0, 1, 128, None, None)
    assert rc != 0 and b"null pointer" in built_lib.irs_last_error()
    rc = built_lib.irs_smooth_zero_order_accumulate(0, prm, 2, 0, None, None, 1, 10, None, None,
                                                    0, 1, 0, 0, 0, 1, 128, None, None)
    assert rc != 0 and b"expects 1 parameters" in built_lib.irs_last_error()
    rc = built_lib.irs_jacobian_xu_batch_f64(3, (ctypes.c_double * 2)(0.05, 0.2), 2, None, None, None, 4, None)
    assert rc != 0 and b"no Jacobian" in built_lib.irs_last_error()
    rc = built_lib.irs_tvlqr_riccati(3, 3, 1, 1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, None)
    assert rc != 0 and b"unsupported TVLQR dims" in built_lib.irs_last_error()


def test_box_penalties_and_bound_helpers(built_lib):
    """Host logic of the bounded TVLQR (irs_mpc_b200/tv_lqr.py) — no GPU needed."""
    from irs_mpc_b200 import tv_lqr
    Q = np.diag([5.0, 5.0, 3.0, 0.1, 0.0])
    R = np.diag([1.0, 0.1])
    dx, du = tv_lqr.box_penalties(Q, R)
    assert dx.shape == (5,) and du.shape == (2,)
    assert np.all(dx >= np.diag(Q)) and np.all(dx >= np.diag(Q).mean() - 1e-15)      # floored at the mean curvature
    assert np.all(du >= 0.5 * np.diag(R)) and np.all(du > 0)
    dx2, du2 = tv_lqr.box_penalties(Q, R, rho0=10.0)
    np.testing.assert_allclose(dx2, 10.0 * dx)
    np.testing.assert_allclose(du2, 10.0 * du)
    # boxes indexed by timestep as in the reference (tv_lqr.py:113-116): a box that is constant over the
    # horizon collapses to one row, a time-varying one keeps a row per timestep, [2, dim] broadcasts
    lo, hi = tv_lqr._box_rows(np.stack((np.tile(-np.ones(3), (6, 1)), np.tile(np.ones(3), (6, 1)))), 6, 3, "x")
    assert np.array_equal(lo, -np.ones(3)) and np.array_equal(hi, np.ones(3))
    varying = np.stack((np.tile(-np.ones(3), (6, 1)), np.tile(np.ones(3), (6, 1))))
    varying[1, 3, 0] = 2.0
    lo, hi = tv_lqr._box_rows(varying, 6, 3, "x")
    assert lo.shape == (6, 3) and hi.shape == (6, 3) and hi[3, 0] == 2.0 and hi[2, 0] == 1.0
    lo, hi = tv_lqr._box_rows(varying, 3, 3, "x")          # the varying row lies beyond the horizon asked for
    assert lo.shape == (3,)
    lo, hi = tv_lqr._box_rows(np.stack((-np.ones(3), np.ones(3))), 4, 3, "x")
    assert lo.shape == (3,)
    with pytest.raises(ValueError):
        tv_lqr._box_rows(varying, 7, 3, "x")               # fewer rows than the horizon
    assert tv_lqr._violates(np.array([1.1]), np.array([-1.0]), np.array([1.0]))
    assert not tv_lqr._violates(np.array([1.0 + 1e-12]), np.array([-1.0]), np.array([1.0]))
    with pytest.raises(NotImplementedError):
        tv_lqr._DimsOnlySystem(3, 3)
    assert tv_lqr._DimsOnlySystem(5, 2).system_id == 1


def test_pipeline_segments_cover_the_horizon_from_the_back(built_lib):
    """Host logic of the pipelined descent (irs_lqr.pipeline_segments): contiguous segments that
    cover [0, T), late timesteps first, about one resident grid of work items each."""
    from irs_mpc_b200.irs_lqr import RESIDENT_BLOCKS, pipeline_segments
    from irs_mpc_b200 import smoothing
    C, _ = smoothing.plan(2, 0, 100, 100000)          # quadrotor, BASELINE.json configs[2]
    segs = pipeline_segments(100, C)
    assert segs == [(75, 100), (50, 75), (25, 50), (0, 25)]
    assert all((hi - lo) * C <= RESIDENT_BLOCKS for lo, hi in segs)
    assert pipeline_segments(100, 1) is None             # too little sampling work to hide anything behind
    assert pipeline_segments(30, 1, forced=3) == [(20, 30), (10, 20), (0, 10)]
    assert pipeline_segments(12, 1, forced=3) is None    # segments shorter than the minimum: one pass
    for T, Cc in ((37, 40), (100, 245), (1000, 3), (64, 30), (60, 25), (200, 13), (33, 50)):
        segs = pipeline_segments(T, Cc)
        assert segs is not None and segs[0][1] == T and segs[-1][0] == 0 and len(segs) <= 8
        assert all(a[0] == b[1] for a, b in zip(segs, segs[1:]))      # contiguous, descending
        assert all(hi - lo >= 8 for lo, hi in segs)
