"""GPU: every randomized-smoothing accumulate kernel against a float64 sum of its own samples, chunk by chunk,
and the chunk reduction, the first-order fit and both zero-order finalize kernels against float64 references of the
same inputs.

The fit-level tests (test_gpu_parity.py, 1e-4 relative) cannot see a kernel that drops, duplicates or re-weights
a few samples: the least-squares fit barely moves.  Here every packed (point, chunk) block the zero-order kernel
writes is compared with `oracle/sample_gram.py: chunk_partials` of the very same rows, formed in float32 from
the library's own deltas (`GaussianSampling.deltas`, or the replayed noise) and its own fp32 dynamics
(`_run_dynamics(..., dtype=torch.float32)`), in units of sum_s |a_si| |b_sj| per entry
(`normalized_error`).  Tolerances, one per engine (oracle/sample_gram.py, shown to reject every mutation
of tests/test_oracle_sample_gram.py by 10x): CUDA cores 2e-6, tensor cores 2e-5.  The tensor-core network of
the learned dynamics also rounds the responses themselves: its bound adds 1e-5 (|f| + |fbar|) per response,
summed like |b| (the single-evaluation tolerance of test_mlp_dynamics.py).

The partial buffer is filled with NaN before every launch and carries a NaN guard after the last block: no NaN
may survive inside, the guard must stay untouched, and entries whose absolute sum is 0 (a sigma = 0 regressor,
the moments of a non-centred three_cart launch) must be exactly 0.

Which test reaches which instantiation through `irs_smooth_zero_order_accumulate` (csrc/api.cu):

| instantiation                                                       | reached by                                   |
|---------------------------------------------------------------------|----------------------------------------------|
| smooth_zero_order_tc_kernel<Sys, 1, kTcPhilox, false>               | test_zero_order_partials_at_sample_edges      |
|   (pendulum, bicycle, quadrotor, three_cart)                        |   [engine 1, antithetic False]               |
| smooth_zero_order_tc_kernel<Sys, 1, kTcPaired, false> (single row)  | ... [engine 1, antithetic True]; the bench   |
|   (three_cart: the DUAL tile, one row per pair)                     |   and batched-MPC shapes                     |
| smooth_zero_order_tc_kernel<ThreeCart, 1, kTcPaired, false/true>    | test_three_cart_projection_modes_partials    |
|   DUAL tile, two rows per pair (projected regressors)               |   [engine 1, antithetic, delta / absolute]   |
| smooth_zero_order_tc_kernel<ThreeCart, 1, kTcPhilox, true>          | test_three_cart_projection_modes_partials    |
|                                                                     |   [engine 1, absolute, not antithetic]       |
| smooth_zero_order_tc_kernel<Sys, 1, kTcReplay, false/true>          | test_replayed_noise_partials,                |
|                                                                     |   test_three_cart_projection_modes_partials  |
|                                                                     |   [replayed absolute points, IRS_CENTERED]   |
| smooth_zero_order_kernel<Sys, 1> (pendulum, bicycle, three_cart)    | every test above at engine 0                 |
| smooth_zero_order_kernel<Quadrotor, 4>                              | every quadrotor case at engine 0             |
| smooth_zero_order_mlp_kernel<Mlp21>                                 | test_mlp_zero_order_partials [tc]            |
| smooth_zero_order_kernel<Mlp21, 1> (IRS_MLP_ENGINE=0)               | test_mlp_zero_order_partials [functor]       |
| smooth_first_order_kernel<Sys> (pendulum, bicycle, quadrotor, MLP)  | test_first_order_means                       |
| reduce_chunks_kernel                                                | test_reduce_chunks_is_the_float64_sum_in_order|
| finalize_zero_order_kernel<Sys, 128> (IRS_FINALIZE_VARIANT=block)  | test_finalize_* (all five): synthetic partials|
| finalize_zero_order_quad_kernel<Sys> (IRS_FINALIZE_VARIANT=quad)   |   and reduced blocks, 1-3 ranks, 1-5 chunks  |
|   (the centred un-shift always takes the block kernel)              | test_finalize_centred_unshift_...            |
| finalize_first_order_kernel<Sys>                                    | test_first_order_means                       |

The engine is chosen with irs_set_gram_engine and restored on leaving the `engine` block.  The persistent
tensor-core grid is sized from the kernel's occupancy, so item counts per block come from the shapes (P = 409,600
at N = 1000 makes every persistent block walk far more than the quadrotor's 64-item nominal batch).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import example_configs as ec          # noqa: E402
from oracle import sample_gram as sg              # noqa: E402

SYSTEMS = ["pendulum", "bicycle", "quadrotor", "three_cart"]
TOL = {0: sg.TOL_CUDA_CORES, 1: sg.TOL_TENSOR_CORES}
MLP_RESPONSE_EPS = 1e-5
N_EDGES = [1, 2, 31, 32, 33, 127, 128, 129, 255, 256, 257, 4095, 4096, 4097, 8193]
# largest normalized partial error seen per engine in this module (printed at its end, -s shows it)
MAX_ERR = {}


@pytest.fixture(scope="module", autouse=True)
def report_max_errors():
    yield
    for k, v in sorted(MAX_ERR.items()):
        print("\nlargest normalized partial error, %s: %.3e" % (k, v))


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


@pytest.fixture(scope="module")
def mlp(api, golden_dir):
    import os
    g = np.load(os.path.join(golden_dir, "mlp_pendulum.npz"))
    return api.MlpDynamics([(g["W1"], g["b1"]), (g["W2"], g["b2"]), (g["W3"], g["b3"])])


def default_engine():
    """The engine the library starts with: IRS_GRAM_ENGINE, read as csrc/api.cu: gram_engine() reads it."""
    import os
    try:
        e = int(os.environ.get("IRS_GRAM_ENGINE", "-1"))
    except ValueError:
        e = 0
    return e if -1 <= e <= 1 else -1


class engine:
    """irs_set_gram_engine for the duration of a with-block; leaving it restores the process's default engine
    (IRS_GRAM_ENGINE or auto), so a suite run with a forced engine keeps it after this module."""

    def __init__(self, e):
        self.e = e

    def __enter__(self):
        from irs_mpc_b200 import _lib
        _lib.call("irs_set_gram_engine", self.e)

    def __exit__(self, *exc):
        from irs_mpc_b200 import _lib
        _lib.call("irs_set_gram_engine", default_engine())


def nominal_points(cfg, n, m, P, seed=7, offset=0.0):
    rng = np.random.default_rng(seed)
    x = np.asarray(cfg["x0"], dtype=np.float64) + 0.3 * rng.standard_normal((P, n))
    u = np.asarray(cfg["u_trj_initial"][0], dtype=np.float64) + 0.3 * rng.standard_normal((P, m))
    if offset:
        x[:, :3] += offset          # three_cart: every cart moved together (the gaps are unchanged)
    if n == 6:
        x[:, 1] = x[:, 0] + 1.0 + 0.05 * rng.standard_normal(P)       # carts apart, a few in contact per chunk
        x[:, 2] = x[:, 1] + 1.0 + 0.05 * rng.standard_normal(P)
    return x, u


def guarded_workspace(s, order, P, N, chunk_samples=0, guard=4096):
    """A Workspace whose partials are NaN and followed by a NaN guard region."""
    import torch
    from irs_mpc_b200 import _device, smoothing
    ws = smoothing.Workspace(s, order, P, N, chunk_samples)
    total = P * ws.C * ws.width
    buf = _device.empty((total + guard,), torch.float32)
    buf.fill_(float("nan"))
    ws.partials = buf[:total].view(P, ws.C, ws.width)
    ws._guard_buf = buf
    return ws


def check_guard(ws):
    import torch
    total = ws.partials.numel()
    g = ws._guard_buf[total:]
    assert bool(torch.isnan(g).all()), "the kernel wrote past the last partial block"


def responses(s, pts, frame, centred, batch):
    """fp32 dynamics of the library at the sample points and at the frame of the nominal response."""
    import torch
    n = s.dim_x
    f = s._run_dynamics(pts[:, :n], pts[:, n:], batch, dtype=torch.float32).astype(np.float32)
    xf, uf = frame
    fb = s._run_dynamics(xf[None], uf[None], batch if centred else False, dtype=torch.float32)[0].astype(np.float32)
    return f, fb


def check_point(s, ws, p, w, pts, frame, centred, N, tol, paired, moments, mlp_eps=0.0):
    """Compare the C blocks of point p with the float64 sums of the kernel's own rows; returns the error."""
    from irs_mpc_b200 import _device
    d = s.dim_x + s.dim_u
    batch = bool(getattr(s, "batch_differs_from_scalar", False))
    f, fb = responses(s, pts, frame, centred, batch)
    rows = sg.paired_rows(w, f, fb) if paired else sg.sample_rows(w, f, fb)
    ref, absref = sg.chunk_partials(rows, N, ws.C, ws.S, d, paired=paired, moments=moments)
    got = _device.to_numpy(ws.partials[p]).astype(np.float64)
    assert got.shape == ref.shape
    assert not np.isnan(got).any(), "a partial entry was never written"
    bound = tol * absref
    if mlp_eps:
        mag = np.hstack((np.abs(w), np.abs(f) + np.abs(fb)[None, :]))
        bound = bound + mlp_eps * sg.chunk_partials(mag, N, ws.C, ws.S, d, paired=paired, moments=moments)[0]
    err = np.abs(got - ref)
    zero = absref == 0
    assert not (err[zero] != 0).any(), "an entry with no contribution is not exactly 0"
    ratio = float(np.max(np.where(zero, 0.0, err / np.where(zero, 1.0, bound))))
    assert ratio <= 1.0, "normalized partial error %.3e over tolerance (ratio %.2f)" % (
        sg.normalized_error(got, ref, absref), ratio)
    return sg.normalized_error(got, ref, absref)


def run_zero_order(api, s, name, N, P, eng, antithetic, chunk_samples=0, projection=None, offset=0.0,
                   seed=99, it=3, stream_id=0, p0=0, i0=0, sigma=None, check=None, replay=None, centered=False):
    """Launch the accumulate on P points and check the listed points (default: all).  replay: [P, N, d] noise
    replayed instead of the Philox stream; centered: it holds absolute points (IRS_CENTERED)."""
    import torch
    from irs_mpc_b200 import _device, sampling, smoothing
    cfg = ec.CONFIGS[name]() if name != "mlp" else ec.pendulum_nn()
    n, m = s.dim_x, s.dim_u
    d = n + m
    x_nom, u_nom = nominal_points(cfg, n, m, P, offset=offset)
    sig0 = np.asarray(cfg["sigma"] if sigma is None else sigma, dtype=np.float64)
    sampler = sampling.GaussianSampling(sig0[:n], sig0[n:], N, power=cfg["power"], seed=seed,
                                        projection=projection, stream_id=stream_id, antithetic=antithetic)
    ws = guarded_workspace(s, smoothing.ZERO_ORDER, P, N, chunk_samples)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    flags = sampler.flags()
    noise = None
    if replay is not None:
        noise = _device.to_device(replay, torch.float32)
        flags = smoothing.FLAG_CENTERED if centered else 0
    if noise is None:
        smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, sigma=sampler.sigma(it), seed=seed, it=it,
                             stream_id=stream_id, p0=p0, i0=i0, flags=flags)
    else:
        smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, noise=noise, flags=flags)
    torch.cuda.synchronize()
    check_guard(ws)
    assert not bool(torch.isnan(ws.partials).any()), "NaN survived in the block region"
    points = range(P) if check is None else check
    centred_capable = name == "three_cart"
    tc = eng == 1 and name != "mlp"
    replay_abs = noise is not None and centered
    paired = tc and antithetic and noise is None and projection is None
    errs = []
    for p in points:
        if noise is None:
            z = sampler.deltas(1, it, t0=p0 + p, i0=i0)[0]
        else:
            z = np.asarray(replay[p], dtype=np.float32)
        project = None
        if projection is not None:
            def project(xp):
                u0 = np.zeros((xp.shape[0], m))
                return sampling.project_samples(s, xp, np.zeros_like(xp), u0, u0)[0]
        w, pts, frame, centred = sg.perturbed_points(x_nom[p], u_nom[p], z, projection, project, replay_abs)
        moments = centred if centred_capable else None
        tol = TOL[1 if (tc or (name == "mlp" and eng == 1)) else 0]
        errs.append(check_point(s, ws, p, w, pts, frame, centred, N, tol, paired, moments,
                                mlp_eps=MLP_RESPONSE_EPS if (name == "mlp" and eng == 1) else 0.0))
    key = ("mlp " if name == "mlp" else "") + ("tensor cores" if eng == 1 else "cuda cores")
    MAX_ERR[key] = max(MAX_ERR.get(key, 0.0), max(errs))
    return ws, max(errs)


# --------------------------------------------------------------------------------------------------
# zero order
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("name", SYSTEMS)
def test_zero_order_partials_at_sample_edges(api, name, eng, antithetic, chunk_samples):
    """Every N edge (ragged rounds, lone pair members, chunk boundaries), P = 3, default and small chunks."""
    s = make_system(api, name)
    with engine(eng):
        for N in N_EDGES:
            run_zero_order(api, s, name, N, 3, eng, antithetic, chunk_samples=chunk_samples)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("name", SYSTEMS)
def test_zero_order_partials_philox_arguments(api, name, eng, antithetic):
    """p0 != 0, an even i0 != 0 (a sample-sharded rank), stream_id != 0, iter > 1, a seed above 2^32."""
    s = make_system(api, name)
    with engine(eng):
        run_zero_order(api, s, name, 4097, 3, eng, antithetic, seed=(1 << 33) + 12345, it=7, stream_id=3, p0=11,
                       i0=8194)


@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("name", ["quadrotor", "three_cart"])
def test_zero_order_partials_at_the_bench_shape(api, name, eng):
    """N = 1e5: 25 chunks of the default plan, the last one partly filled."""
    s = make_system(api, name)
    with engine(eng):
        ws, _ = run_zero_order(api, s, name, 100000, 2, eng, True)
    assert ws.C == 25


@pytest.mark.parametrize("eng", [0, 1])
def test_zero_order_partials_at_the_batched_mpc_shape(api, eng):
    """P = 409,600 quadrotor points of N = 1000 (one 1024-sample chunk each): every persistent block walks
    thousands of items and the 64-item nominal batch rolls over many times.  A spread of points is checked."""
    s = make_system(api, "quadrotor")
    P = 409600
    check = sorted(set([0, 1, 63, 64, 65, P - 1] + list(range(0, P, 4099))))
    with engine(eng):
        ws, _ = run_zero_order(api, s, "quadrotor", 1000, P, eng, True, check=check)
    assert ws.C == 1


@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("name", ["quadrotor", "bicycle"])
def test_zero_sigma_regressor_gives_exact_zeros(api, name, eng):
    """A sigma = 0 regressor: its whole Gram row and column are exactly 0 (checked inside check_point)."""
    s = make_system(api, name)
    sig = np.array(ec.CONFIGS[name]()["sigma"], dtype=np.float64)
    sig[1] = 0.0
    with engine(eng):
        ws, _ = run_zero_order(api, s, name, 4097, 2, eng, True, sigma=sig)
        ws, _ = run_zero_order(api, s, name, 129, 2, eng, False, sigma=sig)


@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("name", SYSTEMS)
def test_replayed_noise_partials(api, name, eng):
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    cfg = ec.CONFIGS[name]()
    rng = np.random.default_rng(3)
    for N in (33, 4097):
        noise = (rng.standard_normal((2, N, n + m)) * cfg["sigma"]).astype(np.float32)
        with engine(eng):
            run_zero_order(api, s, name, N, 2, eng, False, replay=noise)


@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("eng", [0, 1])
@pytest.mark.parametrize("mode", ["none", "delta", "absolute-1e2", "absolute-1e3", "replay-absolute"])
def test_three_cart_projection_modes_partials(api, mode, eng, antithetic):
    """No projection, IRS_PROJECT_DELTA, IRS_PROJECT_ABSOLUTE at |xbar| = 1e2 and 1e3 (centred: the moments are
    checked), and replayed absolute points with IRS_CENTERED."""
    s = make_system(api, "three_cart")
    cfg = ec.CONFIGS["three_cart"]()
    with engine(eng):
        for N in (257, 4097):
            if mode == "none":
                run_zero_order(api, s, "three_cart", N, 2, eng, antithetic)
            elif mode == "delta":
                run_zero_order(api, s, "three_cart", N, 2, eng, antithetic, projection="delta")
            elif mode.startswith("absolute"):
                run_zero_order(api, s, "three_cart", N, 2, eng, antithetic, projection="absolute",
                               offset=float(mode.split("-")[1]))
            else:
                if antithetic:
                    pytest.skip("replayed noise has no antithetic mode")
                x_nom, u_nom = nominal_points(cfg, 6, 2, 2, offset=1e2)
                rng = np.random.default_rng(5)
                z = rng.standard_normal((2, N, 8)) * cfg["sigma"]
                absolute = (np.hstack((x_nom, u_nom))[:, None, :] + z).astype(np.float32)
                run_zero_order(api, s, "three_cart", N, 2, eng, False, offset=1e2, replay=absolute, centered=True)


@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("eng", [0, 1])
def test_mlp_zero_order_partials(api, mlp, eng, chunk_samples, monkeypatch):
    """The tensor-core network (IRS_MLP_ENGINE unset) and the per-thread functor (IRS_MLP_ENGINE=0)."""
    if eng == 0:
        monkeypatch.setenv("IRS_MLP_ENGINE", "0")
    else:
        monkeypatch.delenv("IRS_MLP_ENGINE", raising=False)
    for N in (1, 31, 129, 1535, 1536, 1537, 4097):
        for anti in (False, True):
            run_zero_order(api, mlp, "mlp", N, 3, eng, anti, chunk_samples=chunk_samples)


# --------------------------------------------------------------------------------------------------
# chunk reduction
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 2, 7, 8, 9, 25])
def test_reduce_chunks_is_the_float64_sum_in_order(api, C):
    """[P, C, width] fp32 -> [P, width] fp64, bit for bit the float64 sum in chunk order."""
    import torch
    from irs_mpc_b200 import _device, smoothing
    s = make_system(api, "quadrotor")
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


# --------------------------------------------------------------------------------------------------
# first order
# --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("name", ["pendulum", "bicycle", "quadrotor", "mlp"])
def test_first_order_means(api, mlp, name, chunk_samples):
    """A_t, B_t against the float64 mean of the library's fp32 Jacobians at the identical perturbed points,
    per entry in units of mean_s |J_s| of that entry (a dropped sample moves a varying entry by ~ 1/N of it, a
    scale of max |A| would hide it).  The constant entries come from the fp64 assembly and differ from the fp32
    Jacobians by one rounding."""
    import torch
    from irs_mpc_b200 import _device, sampling, smoothing
    s = mlp if name == "mlp" else make_system(api, name)
    cfg = ec.pendulum_nn() if name == "mlp" else ec.CONFIGS[name]()
    n, m = s.dim_x, s.dim_u
    P = 3
    x_nom, u_nom = nominal_points(cfg, n, m, P)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    for N in N_EDGES + [100000]:
        for anti in (False, True):
            sampler = sampling.GaussianSampling(cfg["sigma"][:n], cfg["sigma"][n:], N, power=cfg["power"], seed=21,
                                                antithetic=anti)
            ws = guarded_workspace(s, smoothing.FIRST_ORDER, P, N, chunk_samples)
            smoothing.accumulate(s, smoothing.FIRST_ORDER, xd, ud, N, ws, sigma=sampler.sigma(2), seed=21, it=2,
                                 flags=sampler.flags())
            At, Bt, ct, status = smoothing.finalize(s, smoothing.FIRST_ORDER, xd, ud, ws, N)
            torch.cuda.synchronize()
            check_guard(ws)
            assert not bool(torch.isnan(ws.partials).any())
            assert int(status.sum().item()) == 0
            AB = np.concatenate((_device.to_numpy(At), _device.to_numpy(Bt)), axis=2)
            for p in range(P):
                z = sampler.deltas(1, 2, t0=p)[0]
                pts = (np.concatenate((x_nom[p], u_nom[p])).astype(np.float32)[None, :] + z).astype(np.float32)
                J = s.jacobian_xu_batch(pts[:, :n], pts[:, n:], dtype=torch.float32)
                mean = J.mean(axis=0)
                scale = np.abs(J).mean(axis=0)
                err = np.abs(AB[p] - mean)
                assert np.all(err[scale == 0] == 0), (N, p)
                r = float(np.max(err[scale > 0] / scale[scale > 0]))
                assert r < sg.TOL_CUDA_CORES, (N, p, anti, r)
                MAX_ERR["first order"] = max(MAX_ERR.get("first order", 0.0), r)


# --------------------------------------------------------------------------------------------------
# finalize, from synthetic partials
# --------------------------------------------------------------------------------------------------
# The fp32 chunk partials and the fp64 reduced blocks are filled directly, so nothing here depends on the sample
# kernels.  (A, B) are compared with a float64 solve of the same summed Gram in the equilibrated coefficients
# (column j times sqrt(G_jj), so a column scaled 1e-3 weighs like the others):
# max |(AB - AB_ref) D| / max |AB_ref D| <= FIN_RTOL * kappa, kappa = the condition number of the
# column-equilibrated Gram.  FIN_RTOL = 1e-12: the kernel sums the C R blocks in its own fixed order and solves by
# Cholesky, numpy sums in another order and solves by LU; on a B200 the two differed by up to 3.9e-14 at kappa 1.7.
# An fp32 step in the sum or the solve would show as ~1e-7, a missing chunk or rank as ~1 / (C R).  The rank rule
# and the zero-column branch are exact.  c_t is compared with cr.affine_offset of the kernel's own (A, B) to 1e-12
# of |f| + |A||xbar| + |B||ubar|.
FIN_RTOL = 1e-12
VARIANTS = ("block", "quad")


def unpack(block, d, n):
    """Packed fp64 block -> (G [d, d], Z^T dF [d, n], first moments)."""
    G, B = np.zeros((d, d)), np.zeros((d, n))
    e = 0
    for i in range(d):
        for j in range(i, d + n):
            if j < d:
                G[i, j] = G[j, i] = block[e]
            else:
                B[i, j - d] = block[e]
            e += 1
    return G, B, block[e:]


def solve_ref(G, B):
    """[A | B] of the normal equations in float64; identically-zero columns get coefficient 0."""
    live = np.diag(G) != 0
    X = np.zeros(B.shape)
    X[live] = np.linalg.solve(G[np.ix_(live, live)], B[live])
    D = 1.0 / np.sqrt(np.diag(G)[live])
    kappa = np.linalg.cond(G[np.ix_(live, live)] * D[:, None] * D[None, :])
    return X.T, kappa


def synthetic_partials(rng, P, C, R, d, n, width, colscale, k=50):
    """fp32 partials [R, P, C, width] of k random samples per (rank, point, chunk), responses near-linear."""
    out = np.zeros((R, P, C, width), dtype=np.float32)
    M = rng.standard_normal((n, d))
    for r in range(R):
        for p in range(P):
            for c in range(C):
                z = rng.standard_normal((k, d)) * colscale
                dF = z @ M.T + 0.01 * rng.standard_normal((k, n))
                blk = sg.pack(z.T @ np.hstack((z, dF)), d, d + n)
                out[r, p, c, :blk.shape[0]] = blk.astype(np.float32)
    return out


def run_finalize(s, x_nom, u_nom, data, path, variant, monkeypatch, n_total, centered=False):
    """data: fp32 partials [R, P, C, width] (path 'partials') or fp64 reduced blocks [R, P, width]."""
    import torch
    from irs_mpc_b200 import _device, smoothing
    R, P = data.shape[0], data.shape[1]
    C = data.shape[2] if path == "partials" else 1
    ws = smoothing.Workspace(s, smoothing.ZERO_ORDER, P, C * 256, chunk_samples=256)
    assert ws.C == C
    ws.centered = centered
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    if path == "partials":
        t = _device.to_device(data, torch.float32)
        kw = dict(partials=t, nranks=R, rank_stride=P * C * ws.width)
    else:
        t = _device.to_device(data, torch.float64)
        kw = dict(reduced=t, nranks=R, rank_stride=P * ws.width)
    monkeypatch.setenv("IRS_FINALIZE_VARIANT", variant)
    try:
        At, Bt, ct, status = smoothing.finalize(s, smoothing.ZERO_ORDER, xd, ud, ws, float(n_total), **kw)
        return (_device.to_numpy(At), _device.to_numpy(Bt), _device.to_numpy(ct),
                _device.to_numpy(status).astype(np.int64))
    finally:
        monkeypatch.delenv("IRS_FINALIZE_VARIANT")


def summed(data, path):
    return data.astype(np.float64).sum(axis=(0, 2)) if path == "partials" else data.sum(axis=0)


def scaled_err(AB, ref, G):
    D = np.sqrt(np.diag(G))
    return float(np.max(np.abs(AB - ref) * D[None, :]) / np.max(np.abs(ref) * D[None, :]))


def check_fit(name, At, Bt, ct, x_nom, u_nom, G, B, p, s):
    from oracle import cpu_restatement as cr
    n = s.dim_x
    AB = np.concatenate((At[p], Bt[p]), axis=1)
    ref, kappa = solve_ref(G, B)
    err = scaled_err(AB, ref, G)
    assert err <= FIN_RTOL * kappa, (p, err, kappa)
    orc = cr.SYSTEMS[name](s.h)
    want = cr.affine_offset(orc, At[p], Bt[p], x_nom[p], u_nom[p])
    scale = np.abs(orc.dynamics(x_nom[p], u_nom[p])) + np.abs(At[p]) @ np.abs(x_nom[p]) + np.abs(Bt[p]) @ np.abs(u_nom[p])
    assert np.all(np.abs(ct[p] - want) <= 1e-12 * scale), p
    return AB[:, :n], ref


@pytest.mark.parametrize("R", [1, 2, 3])
@pytest.mark.parametrize("C", [1, 2, 5])
@pytest.mark.parametrize("name", SYSTEMS)
def test_finalize_matches_float64_solve(api, name, C, R, monkeypatch):
    """1, 2, 5 chunks and 1, 2, 3 ranks, fp32 partials and fp64 reduced blocks, both variants; one regressor
    column is scaled 1e-3 against the others (the bicycle's steer sigma)."""
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    d = n + m
    from irs_mpc_b200 import _lib
    width = _lib.lib().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(100 * C + R)
    P = 3
    x_nom, u_nom = nominal_points(ec.CONFIGS[name](), n, m, P)
    colscale = np.ones(d)
    colscale[d - 2] = 1e-3
    part = synthetic_partials(rng, P, C, R, d, n, width, colscale)
    red = part.astype(np.float64).sum(axis=2)
    for path, data in (("partials", part), ("reduced", red)):
        tot = summed(data, path)
        for variant in VARIANTS:
            At, Bt, ct, status = run_finalize(s, x_nom, u_nom, data, path, variant, monkeypatch, 50 * C * R)
            assert not status.any(), (path, variant, status)
            for p in range(P):
                G, B, _ = unpack(tot[p], d, n)
                check_fit(name, At, Bt, ct, x_nom, u_nom, G, B, p, s)


@pytest.mark.parametrize("name", SYSTEMS)
def test_finalize_zero_sigma_column_gives_exact_zero(api, name, monkeypatch):
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    d = n + m
    from irs_mpc_b200 import _lib
    width = _lib.lib().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(5)
    P, C, R = 3, 2, 2
    x_nom, u_nom = nominal_points(ec.CONFIGS[name](), n, m, P)
    colscale = np.ones(d)
    colscale[1] = 0.0
    part = synthetic_partials(rng, P, C, R, d, n, width, colscale)
    red = part.astype(np.float64).sum(axis=2)
    for path, data in (("partials", part), ("reduced", red)):
        tot = summed(data, path)
        for variant in VARIANTS:
            At, Bt, ct, status = run_finalize(s, x_nom, u_nom, data, path, variant, monkeypatch, 50 * C * R)
            assert not status.any()
            assert np.all(At[:, :, 1] == 0.0), (path, variant)
            for p in range(P):
                G, B, _ = unpack(tot[p], d, n)
                check_fit(name, At, Bt, ct, x_nom, u_nom, G, B, p, s)


@pytest.mark.parametrize("ratio,flagged", [(2e-6, False), (0.5e-6, True)])
@pytest.mark.parametrize("name", ["bicycle", "quadrotor", "three_cart"])
def test_finalize_rank_rule_on_both_sides(api, name, ratio, flagged, monkeypatch):
    """G = L L^T with the last column's squared pivot = ratio * G_kk (documented rule, smooth.cuh: a pivot
    <= 1e-6 G_kk is rank deficient).  L has integer entries, so G is exact in fp32 and the fp64 Cholesky meets
    the pivot exactly."""
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    d = n + m
    from irs_mpc_b200 import _lib
    width = _lib.lib().irs_partial_width(s.system_id, 0)
    k = d - 1
    L = np.eye(d)
    L[k, 0] = round(np.sqrt(1.0 / ratio - 1.0))     # pivot 1, G_kk = L_k0^2 + 1 ~ 1 / ratio
    G = L @ L.T
    assert abs(1.0 / G[k, k] / ratio - 1.0) < 1e-3
    B = np.arange(1, d * n + 1, dtype=np.float64).reshape(d, n) % 7 - 3
    G2 = np.zeros((d, d + n))
    G2[:, :d], G2[:, d:] = G, B
    blk = np.zeros(width)
    packed = sg.pack(G2, d, d + n)
    blk[:packed.shape[0]] = packed
    x_nom, u_nom = nominal_points(ec.CONFIGS[name](), n, m, 1)
    for path, data in (("partials", blk.astype(np.float32)[None, None, None, :]), ("reduced", blk[None, None, :])):
        assert np.array_equal(summed(data, path)[0], blk)
        for variant in VARIANTS:
            At, Bt, ct, status = run_finalize(s, x_nom, u_nom, data, path, variant, monkeypatch, 1000)
            assert status[0] == (1 if flagged else 0), (path, variant)
            if not flagged:
                check_fit(name, At, Bt, ct, x_nom, u_nom, G, B, 0, s)


@pytest.mark.parametrize("name", SYSTEMS)
def test_finalize_flags_only_the_bad_point(api, name, monkeypatch):
    """NaN in one chunk of point 1, +Inf in one chunk of point 3, a Gram that is not PSD at point 4: exactly those
    points get status 1, the others are fitted as usual (both variants, both paths)."""
    s = make_system(api, name)
    n, m = s.dim_x, s.dim_u
    d = n + m
    from irs_mpc_b200 import _lib
    width = _lib.lib().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(9)
    P, C, R = 6, 2, 1
    x_nom, u_nom = nominal_points(ec.CONFIGS[name](), n, m, P)
    part = synthetic_partials(rng, P, C, R, d, n, width, np.ones(d))
    part[0, 1, 1, 3] = np.nan
    part[0, 3, 0, 0] = np.inf
    tot = part.astype(np.float64).sum(axis=(0, 2))
    part[0, 4, 0, 1] = np.float32(3.0 * np.sqrt(tot[4, 0] * tot[4, sg.gram_row_offset(1, d + n)]))   # G_01 > sqrt(G_00 G_11)
    red = part.astype(np.float64).sum(axis=2)
    for path, data in (("partials", part), ("reduced", red)):
        tot = summed(data, path)
        for variant in VARIANTS:
            At, Bt, ct, status = run_finalize(s, x_nom, u_nom, data, path, variant, monkeypatch, 100)
            assert list(status) == [0, 1, 0, 1, 1, 0], (path, variant, status)
            for p in (0, 2, 5):
                G, B, _ = unpack(tot[p], d, n)
                check_fit(name, At, Bt, ct, x_nom, u_nom, G, B, p, s)


@pytest.mark.parametrize("offset", [1e2, 1e3, 3e4])
def test_finalize_centred_unshift_matches_lstsq_on_shifted_samples(api, offset, monkeypatch):
    """three_cart's centred accumulation: the partials hold the Gram of z' = z - xbar and dF' = dF - rho with
    their first moments; the finalize shifts back in fp64 (smooth.cuh, step 1b).  Reference: lstsq of the
    explicitly shifted float64 samples Z = (xbar, ubar) + z', dF = rho + dF', rho = f_batch(2 xbar, 2 ubar) -
    f(xbar, ubar) of the library's fp64 dynamics.  The samples are multiples of 1/4 and 1/64, so every fp32
    partial is exact and the tolerance is the solve's alone (kappa of the SHIFTED Gram)."""
    s = make_system(api, "three_cart")
    n, m = s.dim_x, s.dim_u
    d = n + m
    from irs_mpc_b200 import _lib
    width = _lib.lib().irs_partial_width(s.system_id, 0)
    rng = np.random.default_rng(int(offset))
    P, C, k = 2, 2, 64
    x_nom, u_nom = nominal_points(ec.CONFIGS["three_cart"](), n, m, P, offset=offset)
    rho = s._run_dynamics(2 * x_nom, 2 * u_nom, True) - s._run_dynamics(x_nom, u_nom, False)
    M = rng.integers(-4, 5, (n, d)) * 0.125
    part = np.zeros((1, P, C, width), dtype=np.float32)
    samples = [[] for _ in range(P)]
    for p in range(P):
        for c in range(C):
            z = rng.integers(-4, 5, (k, d)) * 0.25
            dF = z @ M.T + rng.integers(-2, 3, (k, n)) * 2.0 ** -6
            rows = np.hstack((z, dF))
            blk = np.concatenate((sg.pack(z.T @ rows, d, d + n), rows.sum(axis=0)))
            assert np.array_equal(blk.astype(np.float32).astype(np.float64), blk)
            part[0, p, c] = blk
            samples[p].append(rows)
    for variant in VARIANTS:          # a centred fit always takes the block kernel
        At, Bt, ct, status = run_finalize(s, x_nom, u_nom, part, "partials", variant, monkeypatch, C * k,
                                          centered=True)
        assert not status.any()
        for p in range(P):
            rows = np.vstack(samples[p])
            Z = np.concatenate((x_nom[p], u_nom[p]))[None, :] + rows[:, :d]
            dF = rho[p][None, :] + rows[:, d:]
            check_fit("three_cart", At, Bt, ct, x_nom, u_nom, Z.T @ Z, Z.T @ dF, p, s)
            ref = np.linalg.lstsq(Z, dF, rcond=None)[0].T
            AB = np.concatenate((At[p], Bt[p]), axis=1)
            _, kappa = solve_ref(Z.T @ Z, Z.T @ dF)
            assert scaled_err(AB, ref, Z.T @ Z) <= FIN_RTOL * kappa
