"""The learned-dynamics kernels (MlpDynamics) at hidden widths other than the reference network's 100 / 100, against
float64 references of the same operation (GPU tests: run with `-m gpu`).

Four kernel paths change shape with the hidden widths (H1, H2):
- smooth_zero_order_mlp_kernel (csrc/smooth_mlp.cuh): Kp = ceil16(H1 + 1), Np = ceil16(H2), where the first-layer
  operands are staged, 128 or 256 TMEM columns per tile group, one or two groups per block, blocks per SM;
- rollout_mlp_kernel (csrc/tvlqr.cuh): the H1 % 4 and H2 % 4 tails of its summation order;
- Mlp::step_warp (csrc/systems.cuh), the nominal point of the finalize kernel: the same tails, surplus lanes;
- Mlp::hidden / dot_row / jac_var, the per-thread functor of every other kernel.
100 / 100 reaches one layout and no tail at all.  GRID below reaches every layout the launcher can choose (the
restatement `launch_layout` proves it on the CPU) and every residue of H1 % 4 and H2 % 4.

| (H1, H2)   | Kp / Np   | what it exercises                                                              |
|------------|-----------|--------------------------------------------------------------------------------|
| (1, 1)     | 16 / 16   | smallest; both tails = 1 (mod 4); first-layer operands staged separately      |
| (15, 3)    | 16 / 16   | the constant unit in the last column of Kp                                     |
| (31, 17)   | 32 / 32   | largest separate staging; one live unit in the last chunk, read via `vb`      |
| (32, 16)   | 48 / 16   | smallest in-tile staging                                                       |
| (63, 97)   | 64 / 112  | three blocks per SM; tails 3 / 1                                               |
| (100, 100) | 112 / 112 | the reference shape, as control                                                |
| (101, 126) | 112 / 128 | two tile groups of 128 columns; tails 1 / 2                                    |
| (127, 128) | 128 / 128 | Kp full, two groups, even chunk count                                          |
| (128, 1)   | 144 / 16  | 256 TMEM columns, one group                                                    |
| (128, 65)  | 144 / 80  | 256 columns, two groups                                                        |
| (1, 128)   | 16 / 128  | narrow first layer, widest hidden layer                                        |
| (66, 42)   | 80 / 48   | tails 2 / 2 (no other width has H1 = 2 mod 4)                                  |

The networks are random, He-scaled, with each hidden unit's bias placed at a random quantile (0.3 .. 0.7) of its
pre-activation over points drawn like the tests' sample points, so that every unit is active on some points and
inactive on others (test_every_hidden_unit_is_live): a dead unit would hide a dropped or mis-summed tail.

Error bounds scale with the network, not with |f|: the layered forward-error recursion on absolute values
(`forward_error_bound`), gamma(k) = k 2^-24 per float32 sum of k terms, plus EPS_TC per product on the two layers the
tensor cores evaluate (operands split into two bf16 pieces, three products, nominally 2^-16 = 1.5e-5).  EPS_TC comes
from measurement: the largest ratio |f_tc - f_64| / (the recursion's per-product term) over the whole grid was 3.5e-6
on a B200 at a 1000 W power limit (test_tensor_core_response_error prints it); EPS_TC = 1e-5 is 2.9 times that.

Which test reaches which path, at every width of GRID:

| path                                                    | reached by                                           |
|---------------------------------------------------------|------------------------------------------------------|
| smooth_zero_order_mlp_kernel (every layout)             | test_zero_order_partials [tc], _many_points [tc],    |
|                                                         |   test_tensor_core_response_error                    |
| smooth_zero_order_kernel<Mlp21, 1> (IRS_MLP_ENGINE=0)   | test_zero_order_partials [functor], _many_points     |
| Mlp::hidden / dot_row (float32 dynamics batch)          | test_fp32_functor_against_the_float64_twin           |
| smooth_first_order_kernel<Mlp21>, jac_var               | test_first_order_means                               |
| exact_linearize_kernel<Mlp21<double>>                   | test_exact_linearization                             |
| Mlp::step_warp in finalize_zero_order_*                 | test_finalize_nominal_point                          |
| rollout_mlp_kernel<Mlp21, open / closed>                | test_rollouts_and_costs                              |
| the network handle in graph keys and load_params        | test_two_networks_under_cuda_graphs                  |

The largest normalized error of every check is printed at the end of the module (-s shows it).
"""
import gc

import numpy as np
import pytest

from oracle import cpu_restatement as cr
from oracle import sample_gram as sg
from oracle.mlp_ref import MlpOracle

GRID = [(1, 1), (15, 3), (31, 17), (32, 16), (63, 97), (100, 100), (101, 126), (127, 128), (128, 1), (128, 65),
        (1, 128), (66, 42)]
IDS = ["%dx%d" % w for w in GRID]
N_X, N_U = 2, 1
D = N_X + N_U
MAX_HIDDEN = 128
# B200 (sm_100): shared memory per SM and the per-block opt-in limit, in bytes
B200_SMEM_PER_SM = 233472
B200_SMEM_OPTIN = 232448
U32 = 2.0 ** -24                    # unit roundoff of float32
EPS_TC = 1e-5                       # per-product error of the bf16x3 tensor-core layers (module docstring)
SIGMA = np.array([0.3, 0.3, 0.3])   # sample spread (GaussianSampling at it = 1)
NOM_SCALE = 0.6                     # spread of the nominal points
N_LIST = [1, 127, 128, 129, 1535, 1537, 4097]
MAX_ERR = {}


def note(key, v):
    MAX_ERR[key] = max(MAX_ERR.get(key, 0.0), float(v))


@pytest.fixture(scope="module", autouse=True)
def report_max_errors():
    yield
    for k, v in sorted(MAX_ERR.items()):
        print("\nlargest %s: %.3e" % (k, v))


def width_params():
    return pytest.mark.parametrize("hw", [pytest.param(w, id=i) for w, i in zip(GRID, IDS)])


# ------------------------------------------------------------------------------------------------
# the launcher's layout, restated
# ------------------------------------------------------------------------------------------------
def ceil16(v):
    return (v + 15) // 16 * 16


class Layout:
    """csrc/smooth_mlp.cuh: MlpTcLayout."""
    ROWS, K1 = 128, 16

    def __init__(self, h1, h2):
        self.H1, self.H2, self.Kp, self.Np = h1, h2, ceil16(h1 + 1), ceil16(h2)
        self.a_piece = self.ROWS * self.Kp * 2
        self.b_piece = self.Np * self.Kp * 2
        self.a1_piece = self.ROWS * self.K1 * 2
        self.b1_piece = self.Kp * self.K1 * 2
        self.tmem_cols_per_group = 256 if (self.Kp > 128 or self.Np > 128) else 128
        self.stage_bytes = 2 * self.a1_piece + 2 * self.b1_piece
        self.stage_in_tile = self.a_piece >= self.stage_bytes


def tmem_alloc_cols(cols):
    return 128 if cols <= 128 else (256 if cols <= 256 else 512)


K_MAX_GROUPS = 3


def smem_total(L, G):
    """csrc/smooth_mlp.cuh: MlpTcSmem<Mlp21>(L, G).total."""
    width = D * (D + 1) // 2 + D * N_X
    a_stride = 2 * L.a_piece + (0 if L.stage_in_tile else L.stage_bytes)
    o = G * a_stride
    o += 2 * L.b_piece
    o += L.Kp * (D + 1) * 4
    o += (N_X * L.Np + N_X) * 4
    o += 2 * G * MAX_HIDDEN * 4
    o += G * ((N_X + 3) // 4 * 4) * 4
    o += 4 * G * width * 4
    o = (o + 7) // 8 * 8
    return o + 8 * K_MAX_GROUPS + 8


def groups_for(L, limit):
    for g in range(K_MAX_GROUPS, 0, -1):
        if smem_total(L, g) <= limit and g * L.tmem_cols_per_group <= 512:
            return g
    return 0


def launch_layout(h1, h2, per_sm_smem, optin):
    """csrc/api.cu: launch_zero_order_mlp -> (stage in tile, TMEM columns per group, groups per block, blocks per
    SM), or None where the launcher refuses the widths.  Residency is restated from shared memory and TMEM only:
    a register-limited residency (the kernel's launch bounds, 384 threads) is not modelled."""
    L = Layout(h1, h2)
    max_groups = groups_for(L, optin)
    if max_groups < 1:
        return None
    groups = 1 if per_sm_smem // (smem_total(L, 1) + 1024) >= 2 else max_groups
    per_sm = per_sm_smem // (smem_total(L, groups) + 1024)
    per_sm = min(per_sm, 512 // tmem_alloc_cols(groups * L.tmem_cols_per_group))
    return L.stage_in_tile, L.tmem_cols_per_group, groups, max(per_sm, 1)


def regimes(per_sm_smem, optin):
    """Every layout over all 128 x 128 width pairs -> {layout: [pairs]}."""
    out = {}
    for h1 in range(1, MAX_HIDDEN + 1):
        for h2 in range(1, MAX_HIDDEN + 1):
            lay = launch_layout(h1, h2, per_sm_smem, optin)
            assert lay is not None, (h1, h2)
            out.setdefault(lay, []).append((h1, h2))
    return out


def check_coverage(per_sm_smem, optin):
    found = regimes(per_sm_smem, optin)
    reached = {}
    for hw in GRID:
        reached.setdefault(launch_layout(hw[0], hw[1], per_sm_smem, optin), []).append(hw)
    print("\nlayout (stage in tile, TMEM cols / group, groups / block, blocks / SM): pairs, grid widths")
    for lay in sorted(found):
        print("  %s: %5d pairs, grid %s" % (lay, len(found[lay]), reached.get(lay)))
    missing = sorted(set(found) - set(reached))
    assert not missing, "layouts the grid does not reach: %s" % missing
    assert {h1 % 4 for h1, _ in GRID} == {0, 1, 2, 3} and {h2 % 4 for _, h2 in GRID} == {0, 1, 2, 3}
    # the launcher never chooses three groups (DESIGN.md section 3.9)
    assert all(lay[2] <= 2 for lay in found)
    return found


def test_grid_reaches_every_layout_on_b200():
    found = check_coverage(B200_SMEM_PER_SM, B200_SMEM_OPTIN)
    assert len(found) == 7
    # the reference network's layout: staged in the tile, 128 columns, one group, two blocks per SM
    assert launch_layout(100, 100, B200_SMEM_PER_SM, B200_SMEM_OPTIN) == (True, 128, 1, 2)


@pytest.mark.gpu
def test_grid_reaches_every_layout_on_this_device():
    import torch
    prop = torch.cuda.get_device_properties(0)
    check_coverage(prop.shared_memory_per_multiprocessor, prop.shared_memory_per_block_optin)


# ------------------------------------------------------------------------------------------------
# networks, sample points and the float64 twin
# ------------------------------------------------------------------------------------------------
def nominal(P, seed=7):
    rng = np.random.default_rng(seed)
    return NOM_SCALE * rng.standard_normal((P, N_X)), NOM_SCALE * rng.standard_normal((P, N_U))


def proxy_points(seed, count=8192):
    """Points distributed like the tests' sample points: nominal spread plus the sample spread."""
    rng = np.random.default_rng(seed)
    return (np.sqrt(NOM_SCALE ** 2 + SIGMA ** 2) * rng.standard_normal((count, D))).astype(np.float32)


def threshold(z, q):
    """A bias that makes the unit with pre-activations z (minus the bias) active on a fraction ~ 1 - q of them."""
    t = np.quantile(z, q)
    if np.mean(z > t) < 0.1:         # a point mass (ReLU zeros of a narrow first layer) at the quantile
        t = np.quantile(z[z < t], 0.5)
    return -t


def make_weights(h1, h2):
    """He-scaled layers in torch.nn.Linear layout; biases placed so that every hidden unit is live."""
    rng = np.random.default_rng(1000 * h1 + h2)
    pts = proxy_points(100000 + 1000 * h1 + h2).astype(np.float64)
    W1 = rng.standard_normal((h1, D)) * np.sqrt(2.0 / D)
    b1 = np.array([threshold(pts @ W1[j], rng.uniform(0.3, 0.7)) for j in range(h1)])
    a1 = np.maximum(pts @ W1.T + b1, 0.0)
    W2 = rng.standard_normal((h2, h1)) * np.sqrt(2.0 / h1)
    b2 = np.array([threshold(a1 @ W2[j], rng.uniform(0.3, 0.7)) for j in range(h2)])
    W3 = rng.standard_normal((N_X, h2)) * np.sqrt(1.0 / h2)
    b3 = 0.1 * rng.standard_normal(N_X)
    return [np.asarray(v, dtype=np.float32) for v in (W1, b1, W2, b2, W3, b3)]


def twin(hw):
    return MlpOracle(make_weights(*hw), dtype=np.float64)


def forward_error_bound(orc, pts, eps_tc, gamma_scale=1.0):
    """Layered forward-error recursion on absolute values, float64 [B, n]: a bound on |f_computed - f_exact| for a
    float32 evaluation of the network at pts, eps_tc per product on the first two layers (tensor cores)."""
    p = np.asarray(pts, dtype=np.float64)
    H1, H2 = orc.W1.shape[0], orc.W2.shape[0]

    def g(k):
        return gamma_scale * k * U32
    a1 = np.maximum(p @ orc.W1.T + orc.b1, 0.0)
    e1 = (g(D + 1) + eps_tc) * (np.abs(p) @ np.abs(orc.W1).T + np.abs(orc.b1))
    a2 = np.maximum(a1 @ orc.W2.T + orc.b2, 0.0)
    e2 = (g(H1 + 1) + eps_tc) * ((a1 + e1) @ np.abs(orc.W2).T + np.abs(orc.b2)) + e1 @ np.abs(orc.W2).T
    e3 = g(H2 + 1) * ((a2 + e2) @ np.abs(orc.W3).T + np.abs(orc.b3)) + e2 @ np.abs(orc.W3).T
    return e3


def fmaf(a, b, c):
    """float32 fused multiply-add: the product is exact in float64, the sum is rounded once to float64 and once
    to float32 (a double rounding that differs from fmaf only on ties, ~2^-29 of the time)."""
    return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)


def fp32_masks(orc, pts):
    """(a1 > 0, a2 > 0) of the float32 functor (systems.cuh: Mlp::hidden, dot_row's four chains) at pts."""
    W1, b1, W2, b2 = [v.astype(np.float32) for v in (orc.W1, orc.b1, orc.W2, orc.b2)]
    p = np.asarray(pts, dtype=np.float32)
    B, H1, H2 = p.shape[0], W1.shape[0], W2.shape[0]
    s = np.broadcast_to(b1, (B, H1)).copy()
    for q in range(D):
        s = fmaf(W1[None, :, q], p[:, q:q + 1], s)
    a1 = np.maximum(s, np.float32(0))
    acc = [np.broadcast_to(b2, (B, H2)).copy()] + [np.zeros((B, H2), np.float32) for _ in range(3)]
    m4 = H1 & ~3
    for q in range(H1):
        c = q % 4 if q < m4 else 0
        acc[c] = fmaf(W2[None, :, q], a1[:, q:q + 1], acc[c])
    z2 = ((acc[0] + acc[1]).astype(np.float32) + (acc[2] + acc[3]).astype(np.float32)).astype(np.float32)
    return a1 > 0, z2 > 0


def jacobian_bound(orc, masks):
    """|J_fp32 - J_exact| per entry for jac_var's two sums (H2 then H1 terms) over the masked paths."""
    H1, H2 = orc.W1.shape[0], orc.W2.shape[0]
    m1, m2 = [np.asarray(v, dtype=np.float64) for v in masks]
    path = ((np.abs(orc.W3)[None] * m2[:, None, :]) @ np.abs(orc.W2) * m1[:, None, :]) @ np.abs(orc.W1)
    return (H1 + H2 + 2) * U32 * path


@width_params()
def test_every_hidden_unit_is_live(hw):
    """Every hidden unit of both layers is active on some points and inactive on others, on points drawn like the
    sample points of the GPU tests (nominal spread plus sample spread)."""
    orc = twin(hw)
    a1, a2 = orc._hidden(proxy_points(hw[0] * 7 + hw[1]))
    for a in (a1, a2):
        on = (a > 0).mean(axis=0)
        assert np.all(on > 0.02) and np.all(on < 0.98), (hw, on.min(), on.max())


def test_twin_agrees_with_the_float32_oracle_and_the_bound():
    """The float64 twin and the float32 oracle of one network differ by less than the fp32 recursion bound."""
    for hw in GRID:
        w = make_weights(*hw)
        o32, o64 = MlpOracle(w), MlpOracle(w, dtype=np.float64)
        pts = proxy_points(5, 512).astype(np.float64)
        f32, f64 = o32.dynamics_batch(pts[:, :N_X], pts[:, N_X:]), o64.dynamics_batch(pts[:, :N_X], pts[:, N_X:])
        assert np.all(np.abs(f32 - f64) <= forward_error_bound(o64, pts, 0.0)), hw
        masks = fp32_masks(o64, pts)
        J = o64.jacobian_xu_batch(pts[:, :N_X], pts[:, N_X:], masks=masks)
        assert np.all(np.abs(o32.jacobian_xu_batch(pts[:, :N_X], pts[:, N_X:]) - J) <= jacobian_bound(o64, masks)), hw


# ------------------------------------------------------------------------------------------------
# GPU fixtures and helpers
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nets():
    """Every grid network, registered once: hw -> (MlpDynamics, float64 twin)."""
    import torch
    assert torch.cuda.is_available()
    from irs_mpc_b200.systems import MlpDynamics
    out = {}
    for hw in GRID:
        w = make_weights(*hw)
        out[hw] = (MlpDynamics([(w[0], w[1]), (w[2], w[3]), (w[4], w[5])]), MlpOracle(w, dtype=np.float64))
    return out


@pytest.fixture
def mlp_engine(monkeypatch):
    """IRS_MLP_ENGINE for the test: 1 = tensor cores (unset, the default), 0 = the per-thread functor."""
    from irs_mpc_b200 import _graph

    monkeypatch.setattr(_graph, "USE_GRAPHS", False)

    def set_engine(e):
        if e == 0:
            monkeypatch.setenv("IRS_MLP_ENGINE", "0")
        else:
            monkeypatch.delenv("IRS_MLP_ENGINE", raising=False)
    return set_engine


def bounded(err, bound):
    """Largest err / bound; where the bound is 0 (no contributing path or sample) the error must be exactly 0."""
    err, bound = np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64)
    assert not (err[bound == 0] != 0).any(), "an entry with no contribution is not exactly 0"
    live = bound > 0
    return float(np.max(err[live] / bound[live])) if live.any() else 0.0


def functor_f32(s, pts):
    """The library's float32 functor (dynamics batch kernel, fp32) at float32 points."""
    import torch
    p = np.asarray(pts, dtype=np.float64)
    return s._run_dynamics(p[:, :N_X], p[:, N_X:], False, dtype=torch.float32).astype(np.float32)


def run_zero_order(s, orc, N, P, eng, antithetic, chunk_samples=0, seed=99, check=None, live=False):
    """Accumulate on P points and compare every (point, chunk) block with the float64 sums of the rows the kernel
    forms: regressors from the library's own deltas, responses from the library's float32 functor.  The tensor-core
    network rounds its responses differently; its bound adds the recursion of both evaluations per response,
    summed like |b|.  -> (workspace, largest error in units of the bound)."""
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    x_nom, u_nom = nominal(P)
    sampler = sampling.GaussianSampling(SIGMA[:N_X], SIGMA[N_X:], N, power=0.5, seed=seed, antithetic=antithetic)
    ws = tsk.guarded_workspace(s, smoothing.ZERO_ORDER, P, N, chunk_samples)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    smoothing.accumulate(s, smoothing.ZERO_ORDER, xd, ud, N, ws, sigma=sampler.sigma(1), seed=seed, it=1,
                         flags=sampler.flags())
    torch.cuda.synchronize()
    tsk.check_guard(ws)
    assert not bool(torch.isnan(ws.partials).any()), "NaN survived in the block region"
    ratios, masks = [], []
    for p in (range(P) if check is None else check):
        z = sampler.deltas(1, 1, t0=p)[0]
        w, pts, frame, _ = sg.perturbed_points(x_nom[p], u_nom[p], z)
        f = functor_f32(s, pts)
        fb = functor_f32(s, np.concatenate(frame)[None])[0]
        ref, absref = sg.chunk_partials(sg.sample_rows(w, f, fb), N, ws.C, ws.S, D)
        bound = sg.TOL_CUDA_CORES * absref
        if eng == 1:
            resp = forward_error_bound(orc, pts, EPS_TC) + forward_error_bound(orc, pts, 0.0)
            bound = bound + sg.chunk_partials(np.hstack((np.abs(w), resp)), N, ws.C, ws.S, D)[0]
        got = _device.to_numpy(ws.partials[p]).astype(np.float64)
        assert not np.isnan(got).any(), "a partial entry was never written"
        r = bounded(np.abs(got - ref), bound)
        assert r <= 1.0, (p, N, r, sg.normalized_error(got, ref, absref))
        ratios.append(r)
        if live:
            a1, a2 = orc._hidden(pts.astype(np.float64))
            masks.append((a1 > 0, a2 > 0))
    if live:
        for k in range(2):
            on = np.concatenate([mk[k] for mk in masks]).mean(axis=0)
            assert np.all(on > 0) and np.all(on < 1), "a hidden unit is dead on the sample points"
    note("zero-order partial error in units of its bound, %s" % ("tensor cores" if eng else "functor"), max(ratios))
    return ws, max(ratios)


# ------------------------------------------------------------------------------------------------
# the float32 functor and the tensor-core responses against the float64 twin
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@width_params()
def test_fp32_functor_against_the_float64_twin(nets, hw):
    """dynamics_batch (float64 functor over float32 arithmetic) and the float32 dynamics kernel: within the fp32
    recursion bound of the twin at float32 points, and equal to each other."""
    import torch
    s, orc = nets[hw]
    pts = proxy_points(hw[0] + 3 * hw[1], 4096).astype(np.float64)
    want = orc.dynamics_batch(pts[:, :N_X], pts[:, N_X:])
    bound = forward_error_bound(orc, pts, 0.0)
    for got in (s.dynamics_batch(pts[:, :N_X], pts[:, N_X:]),
                s._run_dynamics(pts[:, :N_X], pts[:, N_X:], True, dtype=torch.float32)):
        r = bounded(np.abs(got - want), bound)
        assert r <= 1.0, (hw, r)
        note("fp32 functor error in units of the fp32 recursion", r)
    np.testing.assert_array_equal(s.dynamics_batch(pts[:, :N_X], pts[:, N_X:]), functor_f32(s, pts))


@pytest.mark.gpu
def test_tensor_core_response_error(nets, mlp_engine):
    """The tensor-core network's own responses, read back from one-sample chunks (N = 1: the block holds the
    products w_i r_k, one float32 rounding each), against the float64 twin under the recursion with EPS_TC.  The
    ratio printed is the largest |f_tc - f_64| over the recursion's per-product term: the measured EPS_TC."""
    import torch
    from irs_mpc_b200 import _device, sampling, smoothing
    mlp_engine(1)
    P = 4096
    for hw in GRID:
        s, orc = nets[hw]
        x_nom, u_nom = nominal(P, seed=11)
        sampler = sampling.GaussianSampling(SIGMA[:N_X], SIGMA[N_X:], 1, power=0.5, seed=5, antithetic=False)
        ws = smoothing.Workspace(s, smoothing.ZERO_ORDER, P, 1)
        smoothing.accumulate(s, smoothing.ZERO_ORDER, _device.to_device(x_nom), _device.to_device(u_nom), 1, ws,
                             sigma=sampler.sigma(1), seed=5, it=1, flags=sampler.flags())
        torch.cuda.synchronize()
        blk = _device.to_numpy(ws.partials[:, 0]).astype(np.float64)
        z = sampler.deltas(P, 1)[:, 0]
        frames = np.hstack((x_nom, u_nom)).astype(np.float32)          # the kernel's float32 nominal point
        pts = (frames + z).astype(np.float32)
        fb = functor_f32(s, frames).astype(np.float64)
        w = z.astype(np.float64)
        i = np.argmax(np.abs(w), axis=1)
        rows = np.array([sg.gram_row_offset(k, D + N_X) for k in range(D)])
        resp = np.stack([blk[np.arange(P), rows[i] + (D - i) + k] for k in range(N_X)], axis=1) / w[np.arange(P), i][:, None]
        f_tc = resp + fb
        f64 = orc.dynamics_batch(pts[:, :N_X].astype(np.float64), pts[:, N_X:].astype(np.float64))
        slack = 4 * U32 * (np.abs(resp) + np.abs(fb))            # read-back: the product, the quotient, the sum
        per_product = forward_error_bound(orc, pts, 1.0, gamma_scale=0.0)
        ratio = float(np.max(np.maximum(np.abs(f_tc - f64) - slack, 0.0) / per_product))
        note("tensor-core response error / per-product term (measured EPS_TC)", ratio)
        bound = forward_error_bound(orc, pts, EPS_TC) + slack
        r = bounded(np.abs(f_tc - f64), bound)
        assert r <= 1.0, (hw, r)
    note("EPS_TC", EPS_TC)


# ------------------------------------------------------------------------------------------------
# zero-order partials
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk_samples", [0, 256])
@pytest.mark.parametrize("antithetic", [False, True])
@pytest.mark.parametrize("eng", [1, 0], ids=["tc", "functor"])
@width_params()
def test_zero_order_partials(nets, hw, eng, antithetic, chunk_samples, mlp_engine):
    """Every N edge at P = 3: the item counts P C (3 .. 51) are odd and below the worker count, so two-group blocks
    get uneven and empty workers."""
    s, orc = nets[hw]
    mlp_engine(eng)
    for N in N_LIST:
        run_zero_order(s, orc, N, 3, eng, antithetic, chunk_samples=chunk_samples, live=N == 4097)


@pytest.mark.gpu
@pytest.mark.parametrize("eng", [1, 0], ids=["tc", "functor"])
@width_params()
def test_zero_order_partials_many_points(nets, hw, eng, mlp_engine):
    """P = 2001 points of N = 1537 in chunks of 256: 14,007 items, so every persistent worker walks many; a spread
    of points is checked."""
    s, orc = nets[hw]
    mlp_engine(eng)
    P = 2001
    check = sorted(set([0, 1, 2, 127, 128, 1000, P - 2, P - 1] + list(range(0, P, 331))))
    ws, _ = run_zero_order(s, orc, 1537, P, eng, True, chunk_samples=256, check=check)
    assert ws.C == 7


# ------------------------------------------------------------------------------------------------
# first order, exact linearization, the finalize kernel's nominal point
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@width_params()
def test_first_order_means(nets, hw):
    """A_t, B_t against the float64 mean of the library's fp32 Jacobians at the identical perturbed points (per entry,
    in units of mean |J|), and those Jacobians against the float64 twin with the masks of the float32 activations."""
    import torch
    import test_smoothing_kernels as tsk
    from irs_mpc_b200 import _device, sampling, smoothing
    s, orc = nets[hw]
    P = 3
    x_nom, u_nom = nominal(P)
    xd, ud = _device.to_device(x_nom), _device.to_device(u_nom)
    for N in (129, 4097):
        for anti in (False, True):
            sampler = sampling.GaussianSampling(SIGMA[:N_X], SIGMA[N_X:], N, seed=21, antithetic=anti)
            ws = tsk.guarded_workspace(s, smoothing.FIRST_ORDER, P, N)
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
                J = s.jacobian_xu_batch(pts[:, :N_X], pts[:, N_X:], dtype=torch.float32)
                mean, scale = J.mean(axis=0), np.abs(J).mean(axis=0)
                r = bounded(np.abs(AB[p] - mean), scale)
                assert r < sg.TOL_CUDA_CORES, (N, p, anti, r)
                note("first-order mean error (units of mean |J|)", r)
                masks = fp32_masks(orc, pts)
                p64 = pts.astype(np.float64)
                J64 = orc.jacobian_xu_batch(p64[:, :N_X], p64[:, N_X:], masks=masks)
                r = bounded(np.abs(J - J64), jacobian_bound(orc, masks))
                assert r <= 1.0, (N, p, anti, r)
                note("fp32 Jacobian error in units of its recursion", r)


def make_params(T, x0, u_trj):
    from irs_mpc_b200 import irs_lqr
    from oracle import example_configs as ec
    cfg = ec.pendulum_nn(T=T)
    p = irs_lqr.IrsLqrParameters()
    p.Q, p.Qd, p.R = cfg["Q"], cfg["Qd"], cfg["R"]
    p.x0, p.xd_trj, p.u_trj_initial = x0, cfg["xd_trj"][:T + 1], u_trj
    p.xbound, p.ubound = cfg["xbound"], cfg["ubound"]
    return p


@pytest.mark.gpu
@width_params()
def test_exact_linearization(nets, hw):
    """exact_linearize_kernel<Mlp21<double>> through IrsLqrExact.get_TV_matrices: [A | B] against the twin's Jacobian
    at the float32-rounded point with the float32 masks, c_t against f_64 - A xbar - B ubar, under the recursion."""
    from irs_mpc_b200.irs_lqr import IrsLqrExact
    s, orc = nets[hw]
    T = 37
    x_nom, u_nom = nominal(T + 1, seed=4)
    solver = IrsLqrExact(s, make_params(T, x_nom[0], u_nom[:T]))
    At, Bt, ct = solver.get_TV_matrices(x_nom, u_nom[:T])
    pts = np.hstack((x_nom[:T], u_nom[:T])).astype(np.float32)
    masks = fp32_masks(orc, pts)
    p64 = pts.astype(np.float64)
    J64 = orc.jacobian_xu_batch(p64[:, :N_X], p64[:, N_X:], masks=masks)
    r = bounded(np.abs(np.concatenate((At, Bt), axis=2) - J64), jacobian_bound(orc, masks))
    assert r <= 1.0, r
    note("exact linearization [A|B] error in units of its recursion", r)
    want = orc.dynamics_batch(p64[:, :N_X], p64[:, N_X:]) - np.einsum("tij,tj->ti", At, x_nom[:T]) \
        - np.einsum("tij,tj->ti", Bt, u_nom[:T])
    scale = np.abs(want) + np.einsum("tij,tj->ti", np.abs(At), np.abs(x_nom[:T])) \
        + np.einsum("tij,tj->ti", np.abs(Bt), np.abs(u_nom[:T]))
    r = bounded(np.abs(ct - want), forward_error_bound(orc, pts, 0.0) + 1e-12 * scale)
    assert r <= 1.0, r
    note("exact linearization c_t error in units of its bound", r)


@pytest.mark.gpu
@width_params()
def test_finalize_nominal_point(nets, hw, mlp_engine):
    """c_t of a zero-order fit against cr.affine_offset of the kernel's own (A, B) with f(xbar) from the library's
    fp32 functor, to 1e-12 of its scale: Mlp::step_warp in the finalize kernel must equal the functor bit for bit."""
    from irs_mpc_b200 import sampling
    from irs_mpc_b200.irs_lqr import IrsLqrZeroOrder
    s, _ = nets[hw]
    mlp_engine(1)
    T = 37
    x_nom, u_nom = nominal(T + 1, seed=9)
    sampler = sampling.GaussianSampling(SIGMA[:N_X], SIGMA[N_X:], 1000, seed=13)
    solver = IrsLqrZeroOrder(s, make_params(T, x_nom[0], u_nom[:T]), sampler)
    At, Bt, ct = solver.get_TV_matrices(x_nom, u_nom[:T])
    worst = 0.0
    for t in range(T):
        want = cr.affine_offset(s, At[t], Bt[t], x_nom[t], u_nom[t])
        scale = np.abs(s.dynamics(x_nom[t], u_nom[t])) + np.abs(At[t]) @ np.abs(x_nom[t]) + np.abs(Bt[t]) @ np.abs(u_nom[t])
        assert np.all(np.abs(ct[t] - want) <= 1e-12 * scale), t
        worst = max(worst, float(np.max(np.abs(ct[t] - want) / scale)))
    note("finalize c_t error (rel. to its scale)", worst)


# ------------------------------------------------------------------------------------------------
# rollouts and costs
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("T", [1, 37])
@pytest.mark.parametrize("I", [1, 5])
@width_params()
def test_rollouts_and_costs(nets, hw, I, T):
    """rollout_mlp_kernel: open loop bit-identical to stepping `dynamics` on the host; closed loop equal bit for bit
    to the open-loop replay of the inputs it applied, which equal k + K x to 1e-15 of |k| + |K||x|; costs against
    cr.evaluate_cost to 1e-12; IrsLqr.rollout equal to the host stepping."""
    from irs_mpc_b200 import _device
    from irs_mpc_b200.irs_lqr import IrsLqrExact
    from oracle import example_configs as ec
    s, _ = nets[hw]
    cfg = ec.pendulum_nn(T=T)
    Q, R = cfg["Q"], cfg["R"]
    rng = np.random.default_rng(I * 100 + T + hw[0])
    K = 0.2 * rng.standard_normal((I, T, N_U, N_X))
    k = 0.5 * rng.standard_normal((I, T, N_U))
    x0 = NOM_SCALE * rng.standard_normal((I, N_X))
    xd = cfg["xd_trj"][None, :T + 1] + 0.1 * rng.standard_normal((I, T + 1, N_X))
    u_open = rng.standard_normal((I, T, N_U))
    up = _device.to_device
    dQ, dR, dx0, dxd, dK, dk, du = up(Q), up(R), up(x0), up(xd), up(K), up(k), up(u_open)
    prm, nprm = s._params()

    def open_loop(du_):
        xo, co = _device.empty((I, T + 1, N_X)), _device.empty((I,))
        s.lib.call("irs_rollout_open_loop", s.system_id, prm, nprm, _device.ptr(du_), _device.ptr(dx0),
                   _device.ptr(dxd), (T + 1) * N_X, _device.ptr(dQ), _device.ptr(dR), I, T, _device.ptr(xo),
                   _device.ptr(co), _device.stream_ptr())
        return _device.to_numpy(xo), _device.to_numpy(co)
    xs, us, cost = _device.empty((I, T + 1, N_X)), _device.empty((I, T, N_U)), _device.empty((I,))
    s.lib.call("irs_rollout_closed_loop", s.system_id, prm, nprm, _device.ptr(dK), _device.ptr(dk),
               _device.ptr(dx0), _device.ptr(dxd), (T + 1) * N_X, _device.ptr(dQ), _device.ptr(dR), I, T,
               _device.ptr(xs), _device.ptr(us), _device.ptr(cost), _device.stream_ptr())
    xs, us, cost = _device.to_numpy(xs), _device.to_numpy(us), _device.to_numpy(cost)
    xo, co = open_loop(du)
    dus = up(us)
    xr, cr_ = open_loop(dus)
    for i in range(I):
        np.testing.assert_array_equal(xo[i], cr.rollout(s, x0[i], u_open[i]))
        c = cr.evaluate_cost(xo[i], u_open[i], xd[i], Q, R)
        assert abs(co[i] - c) <= 1e-12 * abs(c), i
        np.testing.assert_array_equal(xr[i], xs[i])
        applied = np.einsum("tij,tj->ti", K[i], xs[i][:T]) + k[i]
        scale = np.abs(k[i]) + np.einsum("tij,tj->ti", np.abs(K[i]), np.abs(xs[i][:T]))
        assert np.all(np.abs(us[i] - applied) <= 1e-15 * scale), i
        c = cr.evaluate_cost(xs[i], us[i], xd[i], Q, R)
        assert abs(cost[i] - c) <= 1e-12 * abs(c), i
        assert abs(cr_[i] - c) <= 1e-12 * abs(c), i
    solver = IrsLqrExact(s, make_params(T, x0[0], u_open[0]))
    np.testing.assert_array_equal(solver.rollout(x0[0], u_open[0]), cr.rollout(s, x0[0], u_open[0]))


# ------------------------------------------------------------------------------------------------
# two networks in one process under CUDA graphs
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_two_networks_under_cuda_graphs(monkeypatch):
    """get_TV_matrices of two widths interleaved past the third call (both replay a captured graph) equals eager
    runs bit for bit; deleting one system leaves the other running, and its released handle is refused."""
    from irs_mpc_b200 import _device, _graph, _lib, sampling
    from irs_mpc_b200.irs_lqr import IrsLqrZeroOrder
    from irs_mpc_b200.systems import MlpDynamics
    monkeypatch.delenv("IRS_MLP_ENGINE", raising=False)
    T, N = 12, 2000
    widths = [(31, 17), (128, 65)]
    trj = {hw: [nominal(T + 1, seed=40 + 2 * j + v) for v in range(2)] for j, hw in enumerate(widths)}

    def system(hw):
        w = make_weights(*hw)
        return MlpDynamics([(w[0], w[1]), (w[2], w[3]), (w[4], w[5])])

    def solver(s, hw):
        x, u = trj[hw][0]
        return IrsLqrZeroOrder(s, make_params(T, x[0], u[:T]),
                               sampling.GaussianSampling(SIGMA[:N_X], SIGMA[N_X:], N, seed=3 + hw[0]))

    monkeypatch.setattr(_graph, "USE_GRAPHS", False)
    eager = {}
    for hw in widths:
        e = solver(system(hw), hw)
        eager[hw] = [e.get_TV_matrices(x, u[:T]) for x, u in trj[hw]]
    monkeypatch.setattr(_graph, "USE_GRAPHS", True)
    systems = {hw: system(hw) for hw in widths}
    solvers = {hw: solver(systems[hw], hw) for hw in widths}
    for call in range(6):
        for hw in widths:
            x, u = trj[hw][call % 2]
            for got, want in zip(solvers[hw].get_TV_matrices(x, u[:T]), eager[hw][call % 2]):
                np.testing.assert_array_equal(got, want)
    assert all(sv._graphs._slots["linearize"][1] is not None for sv in solvers.values()), "no graph was captured"
    gone, kept = widths
    prm_gone = _lib.params_array(systems[gone].device_params())
    del solvers[gone], systems[gone]
    gc.collect()
    for call in range(2):
        x, u = trj[kept][call]
        for got, want in zip(solvers[kept].get_TV_matrices(x, u[:T]), eager[kept][call]):
            np.testing.assert_array_equal(got, want)
    xd, ud, out = _device.to_device(np.zeros((1, N_X))), _device.to_device(np.zeros((1, N_U))), _device.empty((1, N_X))
    with pytest.raises(_lib.IrsCudaError, match="unknown network handle"):
        _lib.call("irs_dynamics_batch_f64", MlpDynamics.system_id, prm_gone[0], prm_gone[1], 0, _device.ptr(xd),
                  _device.ptr(ud), _device.ptr(out), 1, _device.stream_ptr())
