"""Every kernel a user-written system instantiates, on a grid of (n, m) pairs no built-in system has, against float64
references of the same operation at the bars the built-in systems meet (GPU tests: run with `-m gpu`).

A user library (irs_mpc_b200/user_system.py) compiles csrc/api.cu once more around a functor with IRS_USER_N
states and IRS_USER_M inputs, so every hot-path template is instantiated at that shape.  The built-in systems only
reach d = n + m in {3, 7, 8, 16} with (n, m) in {(2,1), (5,2), (6,2), (12,4)}; fit-level tests cannot see a kernel
that drops or re-weights samples or puts a Gram entry in the wrong slot.  The system is oracle/user_grid.py: one
body for every (n, m) in which every state and input has a coefficient of its own, with a float64 numpy twin.

| (n, m)                 | d  | why                                                                          |
|------------------------|----|------------------------------------------------------------------------------|
| (1,1)                  | 2  | smallest; W = 3 padded                                                       |
| (1,7), (3,5), (7,1)    | 8  | last d on the CUDA cores by default; (7,1) has the most G = 1 accumulators   |
| (8,1)                  | 9  | first d on the tensor cores by default; the CUDA-core engine is refused      |
| (4,7)                  | 11 | odd d, n < m                                                                 |
| (10,3)                 | 13 | odd d, n > m, QT = 3 in the quad finalize                                    |
| (15,1), (1,15), (8,8)  | 16 | W = 31; the four-warp CUDA-core split (G = 4)                                |
| (12,4)                 | 16 | built-in dims inside a user library: tiled, packed, segmented Riccati        |

Which test reaches which instantiation of the user library (Sys = UserSystem<R>):

| instantiation                                                  | reached by                                          |
|----------------------------------------------------------------|-----------------------------------------------------|
| dynamics / jacobian batch kernels <float>, <double>            | test_dynamics_and_jacobians                         |
| smooth_zero_order_tc_kernel<Sys, 1, kTcPhilox / kTcPaired>     | test_zero_order_partials_* [tc], every pair         |
|   (dq / nq pieces, kRows up to 64, kNomBatch = 64 for d > 8)   | test_zero_order_partials_many_points [tc, d > 8]    |
| smooth_zero_order_tc_kernel<Sys, 1, kTcReplay>                 | test_replayed_noise_partials [tc]                   |
| smooth_zero_order_kernel<Sys, 1> (d <= 8), <Sys, 4> (d = 16)   | test_zero_order_partials_* [cuda cores]             |
| the CUDA-core refusal for 9 <= d <= 15                         | test_cuda_core_engine_is_refused_for_uneven_rows    |
| reduce_chunks_kernel (user width)                              | test_reduce_chunks_is_the_float64_sum_in_order      |
| finalize_zero_order_kernel<Sys, 128>, the user                 | test_finalize_* [block]                             |
|   make_finalize_tables(IRS_USER_N, IRS_USER_M)                 |                                                     |
| finalize_zero_order_quad_kernel<Sys> (FinalizeQuadCfg, QT)     | test_finalize_* [quad]                              |
| smooth_first_order_kernel<Sys> (NJ = n d up to 240)            | test_first_order_means                              |
|   + finalize_first_order_kernel<Sys>                           |                                                     |
| exact_linearize_kernel<Sys>                                    | test_exact_linearize                                |
| rollout_kernel<Sys, closed / open>                             | test_rollouts_and_costs                             |
| evaluate_cost_kernel<IRS_USER_N, IRS_USER_M>                   | test_rollouts_and_costs                             |
| irs_tvlqr_riccati / linear rollout: the run-time-dimension     | test_lqr_through_the_user_library                   |
|   kernels (non-built-in pairs); tiled, block, warp, packed and |   [every variant of (12,4)]                         |
|   segmented kernels (12,4)                                     |                                                     |
| box_mpc_kernel<UserSystem<double>, true / false>, mpc = 0      | test_box_single_qp_is_certified [both layouts]      |
| box_mpc_kernel<UserSystem<double>, true>, mpc = 1              | test_box_mpc_matches_the_admm_restatement           |
| plan_rows_kernel / plan_check_kernel<IRS_USER_N, IRS_USER_M>   | test_plan_check_flags                               |

Every GPU test is parametrised over the grid, so every row is reached at the nine pairs that are not built in (the
engine rows at the pairs whose d the engine runs).  The largest normalized partial error per engine, and the
largest finalize and rollout errors, are printed at the end of the module (-s shows them).
"""
import concurrent.futures
import contextlib
import ctypes
import time

import numpy as np
import pytest

from irs_mpc_b200 import _lib, user_system
from oracle import cpu_restatement as cr
from oracle import sample_gram as sg
from oracle import user_grid as ug

GRID = [(1, 1), (1, 7), (3, 5), (7, 1), (8, 1), (4, 7), (10, 3), (15, 1), (1, 15), (8, 8), (12, 4)]
IDS = ["%dx%d" % nm for nm in GRID]
N_EDGES = [1, 2, 31, 33, 128, 129, 257, 4097, 8193]
TOL = {0: sg.TOL_CUDA_CORES, 1: sg.TOL_TENSOR_CORES}
ENGINE_NAME = {0: "cuda cores", 1: "tensor cores"}
# largest errors seen in this module (printed at its end)
MAX_ERR = {}
COMPILE = {}


def note(key, v):
    MAX_ERR[key] = max(MAX_ERR.get(key, 0.0), float(v))


@pytest.fixture(scope="module", autouse=True)
def report_max_errors():
    yield
    if COMPILE:
        print("\nuser grid: %d libraries, compile wall time %.1f s (%.1f s summed)"
              % (COMPILE["count"], COMPILE["wall"], COMPILE["summed"]))
    for k, v in sorted(MAX_ERR.items()):
        print("\nlargest %s: %.3e" % (k, v))


def grid_params():
    return pytest.mark.parametrize("nm", [pytest.param(v, id=i) for v, i in zip(GRID, IDS)])


@pytest.fixture(scope="module")
def built():
    """The library of every grid pair, compiled in parallel (or found in the user cache) -> nm: (path, s, hash)."""
    t0 = time.perf_counter()
    with concurrent.futures.ThreadPoolExecutor(len(GRID)) as pool:
        futs = {nm: pool.submit(user_system.build_library, nm[0], nm[1], 1 + len(ug.PARAMS), ug.step_source(),
                                ug.jacobian_source(), "grid_%d_%d" % nm) for nm in GRID}
        out = {nm: f.result() for nm, f in futs.items()}
    summed = sum(v[1] for v in out.values())
    if summed > 0:
        COMPILE.update(count=len(GRID), wall=time.perf_counter() - t0, summed=summed)
    return out


_SYSTEMS = {}


def system(built, nm):
    if nm not in _SYSTEMS:
        _SYSTEMS[nm] = user_system.CudaSourceDynamics(nm[0], nm[1], ug.H, ug.PARAMS, step=ug.step_source(),
                                                      jacobian=ug.jacobian_source(), name="grid_%d_%d" % nm)
        assert _SYSTEMS[nm].library_path == built[nm][0]
    return _SYSTEMS[nm]


def rel(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(float(np.max(np.abs(b))), 1e-300))


# ------------------------------------------------------------------------------------------------
# CPU: the grid compiles, its libraries report their system, the twin is the body's derivative
# ------------------------------------------------------------------------------------------------
@grid_params()
def test_library_loads_and_reports_its_system(built, nm):
    n, m = nm
    lib = _lib.Library.at(built[nm][0])
    h = lib.handle()
    assert h.irs_abi_version() == _lib.ABI_VERSION
    dims = [ctypes.c_int() for _ in range(3)]
    lib.call("irs_system_dims", user_system.USER_SYSTEM_ID, *[ctypes.byref(v) for v in dims])
    d = n + m
    assert [v.value for v in dims] == [n, m, n * d]
    assert h.irs_partial_width(user_system.USER_SYSTEM_ID, 0) == d * (d + 1) // 2 + d * n
    assert h.irs_partial_width(user_system.USER_SYSTEM_ID, 1) == n * d


def test_grid_libraries_are_distinct(built):
    assert len({v[0] for v in built.values()}) == len(GRID)


@grid_params()
def test_twin_jacobian_is_the_derivative_of_the_twin(nm):
    n, m = nm
    orc = ug.GridOracle(n, m)
    rng = np.random.default_rng(n * 17 + m)
    xu = 0.7 * rng.standard_normal((5, n + m))
    J = orc.jacobian_xu_batch(xu[:, :n], xu[:, n:])
    eps = 1e-6
    for j in range(n + m):
        e = np.zeros(n + m)
        e[j] = eps
        fd = (orc.dynamics_batch((xu + e)[:, :n], (xu + e)[:, n:]) -
              orc.dynamics_batch((xu - e)[:, :n], (xu - e)[:, n:])) / (2 * eps)
        assert np.max(np.abs(J[:, :, j] - fd)) < 1e-8, j
    # every input reaches every state with a coefficient of its own sign pattern
    assert np.all(ug.coeffs(n, m) != 0)


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def default_engine():
    import test_smoothing_kernels as tsk
    return tsk.default_engine()


@contextlib.contextmanager
def engine(s, e):
    """The Gram engine of the user library s.lib for the duration of the block (the main library is untouched)."""
    s.lib.call("irs_set_gram_engine", e)
    try:
        yield
    finally:
        s.lib.call("irs_set_gram_engine", default_engine())


def engines(nm):
    """The engines the pair's library runs: the tensor cores always, the CUDA cores where four warps split the
    d rows evenly (d <= 8 by one accumulator group, d = 16 by four)."""
    d = sum(nm)
    return [0, 1] if d <= 8 or d == 16 else [1]


def engine_params():
    return pytest.mark.parametrize("nm,eng", [pytest.param(nm, e, id="%s-%s" % (i, "tc" if e else "ffma"))
                                               for nm, i in zip(GRID, IDS) for e in engines(nm)])


def sigma_of(nm):
    """A distinct sigma per regressor (a mixed-up column changes its scale)."""
    d = sum(nm)
    return 0.05 * (1.0 + 0.15 * np.arange(d))


def nominal(nm, P, seed=7):
    n, m = nm
    rng = np.random.default_rng(seed)
    return 0.5 * rng.standard_normal((P, n)), 0.5 * rng.standard_normal((P, m))


def run_zero_order(s, nm, N, P, eng, antithetic, chunk_samples=0, seed=99, it=3, stream_id=0, p0=0, i0=0,
                   sigma=None, check=None, replay=None):
    """Launch the accumulate of the user library on P points (engine `eng` must be set) and compare the listed
    points (default: all) with the float64 sums of the kernel's own fp32 rows.  Returns (workspace, max error)."""
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    n, m = nm
    x_nom, u_nom = nominal(nm, P)
    sig0 = sigma_of(nm) if sigma is None else np.asarray(sigma, dtype=np.float64)
    sampler = sampling.GaussianSampling(sig0[:n], sig0[n:], N, power=0.5, seed=seed, stream_id=stream_id,
                                        antithetic=antithetic)
    ws = tsk.guarded_workspace(s, smoothing.ZERO_ORDER, P, N, chunk_samples)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    if replay is None:
        smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, sigma=sampler.sigma(it), seed=seed, it=it,
                             stream_id=stream_id, p0=p0, i0=i0, flags=sampler.flags())
    else:
        smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, noise=_device.to_device(replay, torch.float32))
    torch.cuda.synchronize()
    tsk.check_guard(ws)
    assert not bool(torch.isnan(ws.partials).any()), "NaN survived in the block region"
    paired = eng == 1 and antithetic and replay is None
    errs = []
    for p in (range(P) if check is None else check):
        z = sampler.deltas(1, it, t0=p0 + p, i0=i0)[0] if replay is None else np.asarray(replay[p], np.float32)
        w, pts, frame, centred = sg.perturbed_points(x_nom[p], u_nom[p], z)
        errs.append(tsk.check_point(s, ws, p, w, pts, frame, centred, N, TOL[eng], paired, None))
    note("normalized partial error, " + ENGINE_NAME[eng], max(errs))
    return ws, max(errs)


def cfg_of(nm, T):
    """Weights and a target for the rollout, LQR and box tests."""
    n, m = nm
    Q = np.diag(1.0 + 0.1 * np.arange(n))
    R = np.diag(0.1 + 0.05 * np.arange(m))
    xd = np.tile(0.5 * np.sin(1.0 + np.arange(n)), (T + 1, 1))
    return Q, 10.0 * Q, R, xd


# ------------------------------------------------------------------------------------------------
# dynamics and Jacobians
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@grid_params()
def test_dynamics_and_jacobians(built, nm):
    import torch
    n, m = nm
    s, orc = system(built, nm), ug.GridOracle(n, m)
    rng = np.random.default_rng(11)
    x, u = 0.7 * rng.standard_normal((1000, n)), 0.7 * rng.standard_normal((1000, m))
    want = orc.dynamics_batch(x, u)
    for batch in (True, False):
        e = rel(s._run_dynamics(x, u, batch), want)
        assert e <= 1e-12, (batch, e)
        note("fp64 dynamics error (rel. to max |f|)", e)
    assert rel(s.dynamics_batch(x, u), want) <= 1e-12
    assert rel(s.dynamics(x[3], u[3]), want[3]) <= 1e-12
    # the fp32 sample path, at the fp32-rounded points
    x32, u32 = x.astype(np.float32).astype(np.float64), u.astype(np.float32).astype(np.float64)
    e = rel(s._run_dynamics(x32, u32, True, dtype=torch.float32), orc.dynamics_batch(x32, u32))
    assert e <= 1e-5, e
    note("fp32 dynamics error (rel. to max |f|)", e)
    J = orc.jacobian_xu_batch(x, u)
    e = rel(s.jacobian_xu_batch(x, u), J)
    assert e <= 1e-11, e
    note("fp64 Jacobian error (rel. to max |J|)", e)


# ------------------------------------------------------------------------------------------------
# zero-order partials, chunk by chunk
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("antithetic", [False, True])
@engine_params()
def test_zero_order_partials_at_sample_edges(built, nm, eng, antithetic, chunk_samples):
    s = system(built, nm)
    with engine(s, eng):
        for N in N_EDGES:
            run_zero_order(s, nm, N, 3, eng, antithetic, chunk_samples=chunk_samples)


@pytest.mark.gpu
@pytest.mark.parametrize("antithetic", [False, True])
@engine_params()
def test_zero_order_partials_philox_arguments(built, nm, eng, antithetic):
    """p0 != 0, an even i0 != 0, stream_id != 0, iter > 1, a seed above 2^32."""
    s = system(built, nm)
    with engine(s, eng):
        run_zero_order(s, nm, 4097, 3, eng, antithetic, seed=(1 << 33) + 12345, it=7, stream_id=3, p0=11, i0=8194)


@pytest.mark.gpu
@engine_params()
def test_replayed_noise_partials(built, nm, eng):
    s = system(built, nm)
    rng = np.random.default_rng(3)
    for N in (33, 4097):
        noise = (rng.standard_normal((2, N, sum(nm))) * sigma_of(nm)).astype(np.float32)
        with engine(s, eng):
            run_zero_order(s, nm, N, 2, eng, False, replay=noise)


@pytest.mark.gpu
@engine_params()
def test_zero_sigma_regressor_gives_exact_zeros(built, nm, eng):
    """sigma = 0 for the first state, then for the first input: that Gram row and column are exactly 0."""
    s = system(built, nm)
    for col in (0, nm[0]):
        sig = sigma_of(nm)
        sig[col] = 0.0
        with engine(s, eng):
            run_zero_order(s, nm, 4097, 2, eng, True, sigma=sig)
            run_zero_order(s, nm, 129, 2, eng, False, sigma=sig)


@pytest.mark.gpu
@grid_params()
def test_cuda_core_engine_is_refused_for_uneven_rows(built, nm):
    if 0 in engines(nm):
        pytest.skip("the CUDA cores run d = %d" % sum(nm))
    s = system(built, nm)
    with engine(s, 0):
        with pytest.raises(_lib.IrsCudaError, match="evenly"):
            run_zero_order(s, nm, 129, 2, 0, False)


@pytest.mark.gpu
@engine_params()
def test_zero_order_partials_many_points(built, nm, eng):
    """P around the 64-point nominal batch of the tensor-core kernel for d > 8, and ~20,000 points of N = 1000
    (one chunk each) that make every persistent block walk many items; spot-checked there."""
    if sum(nm) <= 8:
        pytest.skip("one nominal point per batch for d <= 8")
    s = system(built, nm)
    with engine(s, eng):
        for P in (1, 63, 64, 65, 129):
            run_zero_order(s, nm, 257, P, eng, True)
        P = 20011
        check = sorted(set([0, 1, 63, 64, 65, 127, 128, P - 1] + list(range(0, P, 1237))))
        ws, _ = run_zero_order(s, nm, 1000, P, eng, True, check=check)
    assert ws.C == 1


# ------------------------------------------------------------------------------------------------
# chunk reduction
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@grid_params()
def test_reduce_chunks_is_the_float64_sum_in_order(built, nm):
    import torch
    from irs_mpc_b200 import _device, smoothing
    s = system(built, nm)
    for C in (1, 3, 9):
        P = 5
        ws = smoothing.Workspace(s, smoothing.ZERO_ORDER, P, 4096 * C, chunk_samples=4096)
        assert ws.C == C
        rng = np.random.default_rng(C)
        host = (rng.standard_normal((P, C, ws.width)) * np.exp(rng.uniform(-20, 20, (P, C, ws.width)))).astype(np.float32)
        ws.partials.copy_(torch.from_numpy(host))
        out = _device.to_numpy(smoothing.reduce_chunks(s, smoothing.ZERO_ORDER, ws))
        want = np.zeros((P, ws.width))
        for c in range(C):
            want += host[:, c].astype(np.float64)
        np.testing.assert_array_equal(out, want)


# ------------------------------------------------------------------------------------------------
# finalize, from synthetic partials
# ------------------------------------------------------------------------------------------------
def check_fit(orc, At, Bt, ct, x_nom, u_nom, G, B, p):
    """[A | B] of point p against the float64 solve (FIN_RTOL kappa, equilibrated) and c_t against
    cr.affine_offset of the twin (1e-12 of |f| + |A||xbar| + |B||ubar|)."""
    import test_smoothing_kernels as tsk
    AB = np.concatenate((At[p], Bt[p]), axis=1)
    ref, kappa = tsk.solve_ref(G, B)
    err = tsk.scaled_err(AB, ref, G)
    assert err <= tsk.FIN_RTOL * kappa, (p, err, kappa)
    note("finalize [A|B] error / (FIN_RTOL kappa)", err / (tsk.FIN_RTOL * kappa))
    want = cr.affine_offset(orc, At[p], Bt[p], x_nom[p], u_nom[p])
    scale = np.abs(orc.dynamics(x_nom[p], u_nom[p])) + np.abs(At[p]) @ np.abs(x_nom[p]) + np.abs(Bt[p]) @ np.abs(u_nom[p])
    assert np.all(np.abs(ct[p] - want) <= 1e-12 * scale), p
    note("finalize c_t error (rel. to its scale)", float(np.max(np.abs(ct[p] - want) / scale)))


def finalize_both(s, x_nom, u_nom, data, path, monkeypatch, n_total):
    """Both finalize variants on the same inputs: they must agree bit for bit.  -> (At, Bt, ct, status)."""
    import test_smoothing_kernels as tsk
    out = [tsk.run_finalize(s, x_nom, u_nom, data, path, v, monkeypatch, n_total) for v in tsk.VARIANTS]
    for a, b in zip(*out):
        assert np.array_equal(a, b, equal_nan=True), path
    return out[0]


@pytest.mark.gpu
@pytest.mark.parametrize("C,R", [(1, 1), (2, 3), (5, 2)])
@grid_params()
def test_finalize_matches_float64_solve(built, nm, C, R, monkeypatch):
    """fp32 partials and fp64 reduced blocks, 1 / 2 / 5 chunks of 1 / 3 / 2 ranks, one regressor column scaled
    1e-3 against the others."""
    import test_smoothing_kernels as tsk
    n, m = nm
    d = n + m
    s, orc = system(built, nm), ug.GridOracle(n, m)
    width = s.lib.handle().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(100 * C + R)
    P = 3
    x_nom, u_nom = nominal(nm, P)
    colscale = 1.0 + 0.1 * np.arange(d)
    colscale[d - 1] = 1e-3
    part = tsk.synthetic_partials(rng, P, C, R, d, n, width, colscale)
    red = part.astype(np.float64).sum(axis=2)
    for path, data in (("partials", part), ("reduced", red)):
        tot = tsk.summed(data, path)
        At, Bt, ct, status = finalize_both(s, x_nom, u_nom, data, path, monkeypatch, 50 * C * R)
        assert not status.any(), (path, status)
        for p in range(P):
            G, B, _ = tsk.unpack(tot[p], d, n)
            check_fit(orc, At, Bt, ct, x_nom, u_nom, G, B, p)


@pytest.mark.gpu
@grid_params()
def test_finalize_zero_sigma_column_gives_exact_zero(built, nm, monkeypatch):
    import test_smoothing_kernels as tsk
    n, m = nm
    d = n + m
    s, orc = system(built, nm), ug.GridOracle(n, m)
    width = s.lib.handle().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(5)
    P, C, R = 3, 2, 2
    x_nom, u_nom = nominal(nm, P)
    for col in (0, n):
        colscale = np.ones(d)
        colscale[col] = 0.0
        part = tsk.synthetic_partials(rng, P, C, R, d, n, width, colscale)
        red = part.astype(np.float64).sum(axis=2)
        for path, data in (("partials", part), ("reduced", red)):
            tot = tsk.summed(data, path)
            At, Bt, ct, status = finalize_both(s, x_nom, u_nom, data, path, monkeypatch, 50 * C * R)
            assert not status.any()
            AB = np.concatenate((At, Bt), axis=2)
            assert np.all(AB[:, :, col] == 0.0), (path, col)
            for p in range(P):
                G, B, _ = tsk.unpack(tot[p], d, n)
                check_fit(orc, At, Bt, ct, x_nom, u_nom, G, B, p)


@pytest.mark.gpu
@grid_params()
def test_finalize_flags_only_the_bad_point(built, nm, monkeypatch):
    """NaN in one chunk of point 1, +Inf in one chunk of point 3, a Gram that is not PSD at point 4."""
    import test_smoothing_kernels as tsk
    n, m = nm
    d = n + m
    s, orc = system(built, nm), ug.GridOracle(n, m)
    width = s.lib.handle().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(9)
    P, C, R = 6, 2, 1
    x_nom, u_nom = nominal(nm, P)
    part = tsk.synthetic_partials(rng, P, C, R, d, n, width, np.ones(d))
    part[0, 1, 1, width - 1] = np.nan
    part[0, 3, 0, 0] = np.inf
    tot = part.astype(np.float64).sum(axis=(0, 2))
    part[0, 4, 0, 1] = np.float32(3.0 * np.sqrt(tot[4, 0] * tot[4, sg.gram_row_offset(1, d + n)]))
    red = part.astype(np.float64).sum(axis=2)
    for path, data in (("partials", part), ("reduced", red)):
        tot = tsk.summed(data, path)
        At, Bt, ct, status = finalize_both(s, x_nom, u_nom, data, path, monkeypatch, 100)
        assert list(status) == [0, 1, 0, 1, 1, 0], (path, status)
        for p in (0, 2, 5):
            G, B, _ = tsk.unpack(tot[p], d, n)
            check_fit(orc, At, Bt, ct, x_nom, u_nom, G, B, p)


# ------------------------------------------------------------------------------------------------
# first order and exact linearization
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk_samples", [0, 256])
@grid_params()
def test_first_order_means(built, nm, chunk_samples):
    """A_t, B_t against the float64 mean of the library's fp32 Jacobians at the identical perturbed points, per
    entry in units of mean_s |J_s| of that entry (the bar of test_smoothing_kernels.py: test_first_order_means)."""
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    n, m = nm
    s = system(built, nm)
    P = 3
    x_nom, u_nom = nominal(nm, P)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    sig = sigma_of(nm)
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
                note("first-order error (per entry, units of mean |J|)", r)


@pytest.mark.gpu
@grid_params()
def test_exact_linearize(built, nm):
    from irs_mpc_b200 import _device
    n, m = nm
    s, orc = system(built, nm), ug.GridOracle(n, m)
    P = 77
    x_nom, u_nom = nominal(nm, P, seed=4)
    At, Bt, ct = _device.empty((P, n, n)), _device.empty((P, n, m)), _device.empty((P, n))
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)      # held: the launch is asynchronous
    prm, nprm = s._params()
    s.lib.call("irs_exact_linearize", s.system_id, prm, nprm, _device.ptr(xd), _device.ptr(ud), P, _device.ptr(At),
               _device.ptr(Bt), _device.ptr(ct), _device.stream_ptr())
    At_o, Bt_o, ct_o = cr.exact_tv_matrices(orc, x_nom, u_nom)
    assert rel(_device.to_numpy(At), At_o) <= 1e-12 and rel(_device.to_numpy(Bt), Bt_o) <= 1e-12
    assert rel(_device.to_numpy(ct), ct_o) <= 1e-12


# ------------------------------------------------------------------------------------------------
# rollouts and costs
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 33])
@pytest.mark.parametrize("I", [1, 3, 65])
@grid_params()
def test_rollouts_and_costs(built, nm, I, T):
    """Closed loop (u = K x + k on the true dynamics) and open loop against the twin, per instance; costs against
    cr.evaluate_cost; irs_evaluate_cost with a shared and a per-instance target."""
    from irs_mpc_b200 import _device
    n, m = nm
    s, orc = system(built, nm), ug.GridOracle(n, m)
    Q, _, R, xd0 = cfg_of(nm, T)
    rng = np.random.default_rng(I * 100 + T)
    K = 0.1 * rng.standard_normal((I, T, m, n))
    k = 0.3 * rng.standard_normal((I, T, m))
    x0 = 0.5 * rng.standard_normal((I, n))
    xd = xd0[None] + 0.1 * rng.standard_normal((I, T + 1, n))
    up = _device.to_device
    u_open = rng.standard_normal((I, T, m))
    # device copies held in names: a temporary could be freed (and its memory handed on) before the launch runs
    dQ, dR, dx0, dxd, dK, dk, du = up(Q), up(R), up(x0), up(xd), up(K), up(k), up(u_open)
    prm, nprm = s._params()
    xs, us, cost = _device.empty((I, T + 1, n)), _device.empty((I, T, m)), _device.empty((I,))
    s.lib.call("irs_rollout_closed_loop", s.system_id, prm, nprm, _device.ptr(dK), _device.ptr(dk),
               _device.ptr(dx0), _device.ptr(dxd), (T + 1) * n, _device.ptr(dQ), _device.ptr(dR), I, T,
               _device.ptr(xs), _device.ptr(us), _device.ptr(cost), _device.stream_ptr())
    xs, us, cost = _device.to_numpy(xs), _device.to_numpy(us), _device.to_numpy(cost)
    xo, co = _device.empty((I, T + 1, n)), _device.empty((I,))
    s.lib.call("irs_rollout_open_loop", s.system_id, prm, nprm, _device.ptr(du), _device.ptr(dx0),
               _device.ptr(dxd), (T + 1) * n, _device.ptr(dQ), _device.ptr(dR), I, T, _device.ptr(xo),
               _device.ptr(co), _device.stream_ptr())
    xo, co = _device.to_numpy(xo), _device.to_numpy(co)
    for i in range(I):
        x_c, u_c = cr.closed_loop_descent(orc, K[i], k[i], x0[i])
        e = max(rel(xs[i], x_c), rel(us[i], u_c))
        assert e <= 1e-12, (i, e)
        note("closed-loop rollout error (rel.)", e)
        c = cr.evaluate_cost(x_c, u_c, xd[i], Q, R)
        assert abs(cost[i] - c) <= 1e-12 * abs(c), i
        x_o = cr.rollout(orc, x0[i], u_open[i])
        e = rel(xo[i], x_o)
        assert e <= 1e-12, (i, e)
        note("open-loop rollout error (rel.)", e)
        c = cr.evaluate_cost(x_o, u_open[i], xd[i], Q, R)
        assert abs(co[i] - c) <= 1e-12 * abs(c), i
    # irs_evaluate_cost on given trajectories, the target shared or per instance
    xt = up(xo)
    for shared in (True, False):
        got = _device.empty((I,))
        s.lib.call("irs_evaluate_cost", n, m, _device.ptr(xt), _device.ptr(du), _device.ptr(dxd),
                   0 if shared else (T + 1) * n, _device.ptr(dQ), _device.ptr(dR), I, T, _device.ptr(got),
                   _device.stream_ptr())
        got = _device.to_numpy(got)
        for i in range(I):
            c = cr.evaluate_cost(xo[i], u_open[i], xd[0 if shared else i], Q, R)
            assert abs(got[i] - c) <= 1e-12 * abs(c), (i, shared)


# ------------------------------------------------------------------------------------------------
# LQR through the user library
# ------------------------------------------------------------------------------------------------
def lqr_problem(nm, I, T, seed):
    n, m = nm
    rng = np.random.default_rng(seed)
    At = 0.9 * np.eye(n) + 0.05 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    x0 = rng.standard_normal((I, n))
    Q, Qd, R, xd = cfg_of(nm, T)
    return At, Bt, ct, x0, Q, Qd, R, xd


@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 7, 40])
@grid_params()
def test_lqr_through_the_user_library(built, nm, T, monkeypatch):
    """irs_tvlqr_riccati and irs_tvlqr_linear_rollout of the user library against cr.tvlqr_riccati and the dense
    KKT solve (bars of test_lqr_kernels.py: 1e-9).  Pairs that are not built in take the run-time-dimension
    kernels and refuse a segment; the (12, 4) library runs every variant of the built-in quadrotor dims, and
    the whole-horizon segment equals the tiled pass bit for bit."""
    import torch
    from oracle import dense_lqr
    from irs_mpc_b200 import _device
    from irs_mpc_b200.tv_lqr import riccati_device
    n, m = nm
    s = system(built, nm)
    I = 9
    At, Bt, ct, x0, Q, Qd, R, xd = lqr_problem(nm, I, T, 31 * n + m + T)
    up = _device.to_device
    d = [up(v) for v in (At, Bt, ct, Q, Qd, R, xd, x0)]
    Ko, ko = zip(*[cr.tvlqr_riccati(At[i], Bt[i], ct[i], Q, Qd, R, xd) for i in range(I)])
    Ko, ko = np.stack(Ko), np.stack(ko)
    u_dense = [dense_lqr.solve(At[i], Bt[i], ct[i], Q, Qd, R, x0[i], xd)[1] for i in (0, I - 1)]
    variants = [None, "block", "warp", "packed"] if nm == (12, 4) else [None]
    out = {}
    for v in variants:
        if v is None:
            monkeypatch.delenv("IRS_TVLQR_VARIANT", raising=False)
        else:
            monkeypatch.setenv("IRS_TVLQR_VARIANT", v)
        K, k, status = riccati_device(*d[:7], 0, lib=s.lib)
        assert np.all(_device.to_numpy(status) == 0), v
        Kn, kn = _device.to_numpy(K), _device.to_numpy(k)
        assert rel(Kn, Ko) < 1e-9 and rel(kn, ko) < 1e-9, (v, rel(Kn, Ko), rel(kn, ko))
        note("Riccati gain error (rel.)", max(rel(Kn, Ko), rel(kn, ko)))
        xs, us = _device.empty((I, T + 1, n)), _device.empty((I, T, m))
        s.lib.call("irs_tvlqr_linear_rollout", n, m, _device.ptr(d[0]), _device.ptr(d[1]), _device.ptr(d[2]),
                   _device.ptr(K), _device.ptr(k), _device.ptr(d[7]), I, T, _device.ptr(xs), _device.ptr(us),
                   _device.stream_ptr())
        us = _device.to_numpy(us)
        for j, i in enumerate((0, I - 1)):
            assert rel(us[i], u_dense[j]) < 1e-9, (v, i, rel(us[i], u_dense[j]))
        out[v] = (Kn, kn)
    monkeypatch.delenv("IRS_TVLQR_VARIANT", raising=False)
    K, k = _device.empty((I, T, m, n)), _device.empty((I, T, m))
    status = _device.empty((I,), torch.int32)

    def segment():
        s.lib.call("irs_tvlqr_riccati_segment", n, m, *[_device.ptr(v) for v in d[:7]], 0, I, T, 0, T, None,
                   _device.ptr(K), _device.ptr(k), _device.ptr(status), _device.stream_ptr())
    if nm in user_system.BUILTIN_PAIRS:
        segment()
        assert np.all(_device.to_numpy(status) == 0)
        assert np.array_equal(_device.to_numpy(K), out[None][0]) and np.array_equal(_device.to_numpy(k), out[None][1])
    else:
        with pytest.raises(_lib.IrsCudaError, match="segmented Riccati"):
            segment()


# ------------------------------------------------------------------------------------------------
# box-constrained QP and the plan check
# ------------------------------------------------------------------------------------------------
def box_api():
    import test_box_qp_kernels as tbq
    return tbq, tbq.Api()


@pytest.mark.gpu
@grid_params()
def test_box_single_qp_is_certified(built, nm):
    """box_mpc_kernel<UserSystem<double>> with mpc = 0, certified by oracle/box_kkt.py, with the per-step matrices
    in shared memory (T = 12) and, where the state is large enough for it to bite at a short horizon, without
    (T = T_cache + 1: box_mpc_smem_bytes(T, true) > 200 KiB)."""
    from oracle import box_kkt as bk
    tbq, api = box_api()
    n, m = nm
    s = system(built, nm)
    Ts = [12]
    if tbq.t_cache(n, m) < 150:
        Ts.append(tbq.t_cache(n, m) + 1)
    for T in Ts:
        for box in ("input", "both"):
            p = bk.make_problem(n, m, T, box, "dense", I=2, seed=7 * n + m + T)
            x, u, cost, status, iters = tbq.solve(api, p, system=s)
            for i in range(2):
                tbq.check_instance(p, i, x, u, cost, status, iters, margins=False)


@pytest.mark.gpu
@grid_params()
def test_box_mpc_matches_the_admm_restatement(built, nm):
    """box_mpc_kernel<UserSystem<double>> with mpc = 1 (the closed loop on the true dynamics) against
    oracle/box_tvlqr.py: mpc_box_descent on the twin: the true dynamics at 1e-12, the first input at the
    certificate bar, the whole loop at 1e-5 (differences below the bar grow along the loop)."""
    from oracle import box_kkt as bk
    from oracle import box_tvlqr as bq
    tbq, api = box_api()
    n, m = nm
    s, orc = system(built, nm), ug.GridOracle(n, m)
    T, I = 12, 2
    Q, Qd, R, xd = cfg_of(nm, T)
    rng = np.random.default_rng(n + 20 * m)
    u_init = 0.3 * rng.standard_normal((T, m))
    x_init = cr.rollout(orc, np.zeros(n), u_init)
    At, Bt, ct = cr.exact_tv_matrices(orc, x_init, u_init)
    K0, k0 = cr.tvlqr_riccati(At, Bt, ct, Q, Qd, R, xd)
    x0 = 0.3 * rng.standard_normal((I, n))
    u_free = np.concatenate([cr.closed_loop_descent(orc, K0, k0, x0[i])[1] for i in range(I)])
    uc = np.median(u_free, axis=0)
    ua = np.quantile(np.abs(u_free - uc), 0.8, axis=0)
    p = dict(At=np.tile(At, (I, 1, 1, 1)), Bt=np.tile(Bt, (I, 1, 1, 1)), ct=np.tile(ct, (I, 1, 1)), xd=xd[None],
             x0=x0, Q=Q, Qd=Qd, R=R, xlo=np.full(n, -bk.BIG), xhi=np.full(n, bk.BIG), ulo=uc - ua, uhi=uc + ua,
             n=n, m=m, T=T, I=I, shared_xd=True)
    gains = (np.tile(K0, (I, 1, 1, 1)), np.tile(k0, (I, 1, 1)))
    x, u, cost, status, iters = tbq.solve(api, p, mpc=True, system=s, gains=gains)
    assert np.all(status == 0)
    assert np.any(iters > 0), "no QP had an active bound"
    for i in range(I):
        for t in range(T):
            f = orc.dynamics(x[i][t], u[i][t])
            assert np.max(np.abs(x[i][t + 1] - f)) <= 1e-12 * max(1.0, np.max(np.abs(f))), (i, t)
        assert abs(cost[i] - cr.evaluate_cost(x[i], u[i], xd, Q, R)) <= 1e-12 * abs(cost[i])
        xo, uo, _ = bq.mpc_box_descent(orc, At, Bt, ct, Q, Qd, R, x0[i], xd, p["xlo"], p["xhi"], p["ulo"], p["uhi"],
                                       gains0=(K0, k0))
        assert np.max(np.abs(u[i][0] - uo[0])) <= tbq.BAR * max(1.0, np.max(np.abs(uo[0]))), i
        assert np.max(np.abs(u[i] - uo)) <= 1e-5 * max(1.0, np.max(np.abs(uo))), i
        assert np.max(np.abs(x[i] - xo)) <= 1e-5 * max(1.0, np.max(np.abs(xo))), i
        note("bounded MPC input error against the restatement (rel.)", rel(u[i], uo))


@pytest.mark.gpu
@grid_params()
def test_plan_check_flags(built, nm):
    """irs_tvlqr_plan_check of the user library against a numpy evaluation of every plan: a box that holds every
    plan flags nothing; moving one bound of the first state, the last state, the first input and the last input
    1e-6 past instance i's extreme value flags instance i only (rows computed by the check, and by plan_rows)."""
    import torch
    import test_lqr_kernels as tlq
    from irs_mpc_b200 import _device
    from irs_mpc_b200.tv_lqr import BOUND_TOL
    n, m = nm
    s = system(built, nm)
    I, T = 3, 12
    rng = np.random.default_rng(n * 10 + m)
    At = 0.9 * np.eye(n) + 0.05 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    K = 0.1 * rng.standard_normal((I, T, m, n))
    k = 0.1 * rng.standard_normal((I, T, m))
    x_trj = rng.standard_normal((I, T + 1, n))
    values, _ = tlq.plans(At, Bt, ct, K, k, x_trj)
    vmax, vmin = np.nanmax(values, axis=(1, 2)), np.nanmin(values, axis=(1, 2))
    lo0, hi0 = vmin.min(axis=0) - 1.0, vmax.max(axis=0) + 1.0
    up = _device.to_device
    d = [up(v) for v in (At, Bt, ct, K, k, x_trj)]
    scratch = _device.empty((I, T, n + m, n + 1))
    violated = _device.empty((I,), torch.int32)
    s.lib.call("irs_tvlqr_plan_rows", n, m, *[_device.ptr(v) for v in d[:5]], I, T, _device.ptr(scratch),
               _device.stream_ptr())

    def check(lo, hi, rows_ready):
        dlo, dhi = up(lo), up(hi)
        s.lib.call("irs_tvlqr_plan_check", n, m, *[_device.ptr(v) for v in d], _device.ptr(dlo[:n]),
                   _device.ptr(dhi[:n]), _device.ptr(dlo[n:]), _device.ptr(dhi[n:]), BOUND_TOL, I, T, rows_ready,
                   _device.ptr(violated), _device.ptr(scratch), _device.stream_ptr())
        return _device.to_numpy(violated)

    for rows_ready in (1, 0):
        assert np.array_equal(check(lo0, hi0, rows_ready), np.zeros(I, np.int32))
    for c in sorted({0, n - 1, n, n + m - 1}):
        for side in ("lo", "hi"):
            ext = vmin[:, c] if side == "lo" else vmax[:, c]
            i = int(np.argmin(ext) if side == "lo" else np.argmax(ext))
            lo, hi = lo0.copy(), hi0.copy()
            if side == "lo":
                lo[c] = ext[i] + BOUND_TOL + 1e-6
            else:
                hi[c] = ext[i] - BOUND_TOL - 1e-6
            want = tlq.flags(values, lo, hi, BOUND_TOL)
            assert want[i] == 1
            for rows_ready in (1, 0):
                assert np.array_equal(check(lo, hi, rows_ready), want), (c, side, rows_ready)
