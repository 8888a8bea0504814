"""Every fp64 Riccati kernel variant against float64 references, through the C ABI (run with `-m gpu`).

References: the recursion oracle `cr.tvlqr_riccati` (gains, value-function Hessians) and the dense KKT
solve of the literal QP, `oracle/dense_lqr.py`, which shares none of the recursion's assumptions
(minimiser u*, checked through `irs_tvlqr_linear_rollout`, the `solve_tvlqr` path).

Which parametrisation reaches which kernel (`irs_tvlqr_riccati_impl` in csrc/api.cu; the variant is picked
with IRS_TVLQR_VARIANT, read at every call):

| label           | how it is selected                                | kernel                                   | dims           |
|-----------------|---------------------------------------------------|------------------------------------------|----------------|
| `tiled`         | `block` (or default), even n, m                   | `tvlqr_riccati_tiled_kernel`             | (6,2) (12,4)   |
| `generic-block` | `block`, odd dims; `irs_tvlqr_riccati_ex` for even | `tvlqr_riccati_kernel<n,m,256>`         | all four       |
| `generic-warp`  | `warp`                                            | `tvlqr_riccati_kernel<n,m,32>`           | all four       |
| `packed`        | `packed`                                          | `tvlqr_riccati_packed_kernel<12,4>`      | (12,4)         |
| segments        | `irs_tvlqr_riccati_segment`                       | `tvlqr_riccati_tiled_kernel`, t_hi > 0   | (6,2) (12,4)   |

`test_variants_match_the_oracle_and_the_dense_qp` runs every row of the table for every dims, horizon and
weight kind at the instance counts where the variant's grouping changes (warp: 4 instances per block;
packed: 2 per warp, 8 per block).  `test_default_dispatch_of_many_instances` lets the dispatch choose at
300 instances (pendulum and bicycle -> `generic-warp`) and at 1030 (quadrotor -> `packed`).

Weights are used as given: a non-symmetric Q, Qd or R describes the same problem as its symmetric part,
and every kernel must return that problem's minimiser.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import cpu_restatement as cr          # noqa: E402
from oracle import dense_lqr                      # noqa: E402

DIMS = [(2, 1), (5, 2), (6, 2), (12, 4)]
HORIZONS = [1, 2, 7, 100]
WEIGHTS = ["diag", "dense", "nonsym", "illcond", "scale+30", "scale-30"]
I_BLOCK = (1, 2, 17)
I_WARP = (1, 3, 4, 5)
I_PACKED = (1, 2, 3, 7, 8, 9, 17)
I_MAX = 17
EPS = np.finfo(np.float64).eps


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


class Api:
    def __init__(self):
        import torch
        from irs_mpc_b200 import _device, _lib
        from irs_mpc_b200.tv_lqr import BOUND_TOL
        self.torch, self.dev, self.lib, self.BOUND_TOL = torch, _device, _lib, BOUND_TOL

    def up(self, a):
        return self.dev.to_device(np.ascontiguousarray(a, dtype=np.float64))

    def np(self, t):
        return self.dev.to_numpy(t)


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    import irs_mpc_b200.all  # noqa: F401
    return Api()


def variants(n, m):
    """(label, IRS_TVLQR_VARIANT, through irs_tvlqr_riccati_ex, instance counts) of every kernel for (n, m)."""
    if n % 2 or m % 2:
        return [("generic-block", "block", False, I_BLOCK), ("generic-warp", "warp", False, I_WARP)]
    out = [("tiled", "block", False, I_BLOCK), ("generic-block", "block", True, I_BLOCK),
           ("generic-warp", "warp", False, I_WARP)]
    if (n, m) == (12, 4):
        out.append(("packed", "packed", False, I_PACKED))
    return out


def spd(rng, d, lo=0.5):
    M = rng.standard_normal((d, d))
    return M.dot(M.T) / d + lo * np.eye(d)


def problem(n, m, T, kind, I=I_MAX, seed=0):
    """I instances of a random affine problem and weights of the given kind.  Returns a dict; `ref` holds
    the weights the references use (for the scaled kinds: the unscaled ones, the minimiser is the same)."""
    rng = np.random.default_rng(seed)
    At = np.eye(n) + 0.1 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    xd = rng.standard_normal((I, T + 1, n))
    x0 = rng.standard_normal((I, n))
    if kind == "diag":
        Q, Qd, R = np.diag(rng.uniform(0.5, 2, n)), np.diag(rng.uniform(5, 20, n)), np.diag(rng.uniform(0.5, 2, m))
    elif kind == "illcond":
        # state weights over 1e-4 .. 1e4, inputs of authority 1 .. 1e-3 and an R too small to lift the weak
        # direction: cond(H) = 1e7 .. 1e8 for m >= 2 (m = 1: H is a scalar)
        Q = np.diag(rng.permutation(np.logspace(-4, 4, n)))
        Qd = np.diag(rng.permutation(np.logspace(-4, 4, n)))
        R = 1e-8 * np.diag(np.logspace(0, 4, m))
        Bt = Bt * np.logspace(0, -3, m)
    else:
        Q, Qd, R = spd(rng, n), 10 * spd(rng, n), spd(rng, m)
        if kind == "nonsym":      # the same kind of SPD symmetric parts plus skew parts of comparable size
            Q, Qd, R = (W + (lambda S: S - S.T)(rng.standard_normal(W.shape)) for W in (Q, Qd, R))
    ref = (Q, Qd, R)
    if kind.startswith("scale"):
        s = 10.0 ** int(kind[5:])
        Q, Qd, R = s * Q, s * Qd, s * R
    return dict(At=At, Bt=Bt, ct=ct, Q=Q, Qd=Qd, R=R, xd=xd, x0=x0, ref=ref, n=n, m=m, T=T)


def xd_of(p, shared):
    return p["xd"][:1] if shared else p["xd"]


def upload(api, p, shared):
    d = {k: api.up(p[k]) for k in ("At", "Bt", "ct", "Q", "Qd", "R", "x0")}
    d["xd"] = api.up(xd_of(p, shared))
    d["xd_stride"] = 0 if shared else (p["T"] + 1) * p["n"]
    return d


def riccati(api, d, n, m, I, T, env, ex, monkeypatch, Q=None, Qd=None, R=None):
    """One backward pass of the first I instances -> device (K, k, status, Hinv, P) (Hinv, P: only with ex)."""
    dev, lib = api.dev, api.lib
    monkeypatch.setenv("IRS_TVLQR_VARIANT", env)
    K, k = dev.empty((I, T, m, n)), dev.empty((I, T, m))
    status = api.torch.full((I,), -1, dtype=api.torch.int32, device=K.device)
    Q, Qd, R = (d[key] if v is None else v for key, v in (("Q", Q), ("Qd", Qd), ("R", R)))
    head = (n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(Q), dev.ptr(Qd), dev.ptr(R),
            dev.ptr(d["xd"]), d["xd_stride"], I, T, dev.ptr(K), dev.ptr(k), dev.ptr(status))
    Hinv = P = None
    if ex:
        Hinv, P = dev.empty((I, T, m, m)), dev.empty((I, T + 1, n, n))
        lib.call("irs_tvlqr_riccati_ex", *head, dev.ptr(Hinv), dev.ptr(P), dev.stream_ptr())
    else:
        lib.call("irs_tvlqr_riccati", *head, dev.stream_ptr())
    monkeypatch.delenv("IRS_TVLQR_VARIANT")
    api.torch.cuda.synchronize()
    return K, k, status, Hinv, P


def linear_rollout(api, d, n, m, I, T, K, k):
    dev = api.dev
    xs, us = dev.empty((I, T + 1, n)), dev.empty((I, T, m))
    api.lib.call("irs_tvlqr_linear_rollout", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(K),
                 dev.ptr(k), dev.ptr(d["x0"]), I, T, dev.ptr(xs), dev.ptr(us), dev.stream_ptr())
    return api.np(us)


def oracle(p, shared, I, hessians=False):
    Q, Qd, R = p["ref"]
    xd = xd_of(p, shared)
    out = [cr.tvlqr_riccati(p["At"][i], p["Bt"][i], p["ct"][i], Q, Qd, R, xd[0 if shared else i],
                            return_hessians=hessians) for i in range(I)]
    return [np.stack([o[j] for o in out]) for j in range(len(out[0]))]


def tolerances(p, kind, H):
    """(against the oracle / the dense QP, between variants).  1e-9 and 1e-10, except for the ill-conditioned
    weights: the forward error of a solve with H grows with cond(H) times the unit round-off; 1e-15 cond(H)
    (about 10 u cond(H)) and a tenth of that between variants."""
    if kind != "illcond":
        return 1e-9, 1e-10
    cond = max(float(np.linalg.cond(h)) for h in H.reshape(-1, p["m"], p["m"]))
    return max(1e-9, 1e-15 * cond), max(1e-10, 1e-16 * cond)


# ------------------------------------------------------------------------------------------------
# gains of every variant: oracle, dense QP, each other
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", WEIGHTS)
@pytest.mark.parametrize("T", HORIZONS)
@pytest.mark.parametrize("n,m", DIMS)
def test_variants_match_the_oracle_and_the_dense_qp(api, n, m, T, kind, monkeypatch):
    p = problem(n, m, T, kind, seed=1000 * n + 100 * m + T + WEIGHTS.index(kind))
    dense_cache = {}

    def dense_u(shared, i):
        if (shared, i) not in dense_cache:
            Q, Qd, R = p["ref"]
            xd = xd_of(p, shared)[0 if shared else i]
            dense_cache[shared, i] = dense_lqr.solve(p["At"][i], p["Bt"][i], p["ct"][i], Q, Qd, R, p["x0"][i], xd)[1]
        return dense_cache[shared, i]

    for shared in (False, True):
        d = upload(api, p, shared)
        Ko, ko, _, Ho = oracle(p, shared, I_MAX, hessians=True)
        tol, tol_x = tolerances(p, kind, Ho)
        full = {}
        for label, env, ex, counts in variants(n, m):
            for I in counts:
                K, k, status, _, _ = riccati(api, d, n, m, I, T, env, ex, monkeypatch)
                Kn, kn = api.np(K), api.np(k)
                where = (label, I, "shared xd" if shared else "xd per instance")
                assert np.all(api.np(status) == 0), where
                assert rel_err(Kn, Ko[:I]) < tol and rel_err(kn, ko[:I]) < tol, \
                    where + (rel_err(Kn, Ko[:I]), rel_err(kn, ko[:I]))
            full[label] = (Kn, kn)
            # u* of the linear model from x0: the solve_tvlqr path, against the dense KKT solve
            us = linear_rollout(api, d, n, m, I, T, K, k)
            for i in ((0,) if T > 7 else (0, I - 1)):
                assert rel_err(us[i], dense_u(shared, i)) < tol, where + (i, rel_err(us[i], dense_u(shared, i)))
        # the variants against each other on the instances they share
        labels = list(full)
        for a in labels[1:]:
            c = min(full[a][0].shape[0], full[labels[0]][0].shape[0])
            assert rel_err(full[a][0][:c], full[labels[0]][0][:c]) < tol_x, (a, labels[0])
            assert rel_err(full[a][1][:c], full[labels[0]][1][:c]) < tol_x, (a, labels[0])


@pytest.mark.parametrize("n,m,I", [(2, 1, 300), (5, 2, 300), (6, 2, 300), (12, 4, 300), (12, 4, 1030)])
def test_default_dispatch_of_many_instances(api, n, m, I, monkeypatch):
    """The dispatch's own choice (no IRS_TVLQR_VARIANT): pendulum and bicycle above 296 instances take the
    warp kernel, the quadrotor above 1000 the packed one; gains against the oracle and the block kernel."""
    T = 7
    p = problem(n, m, T, "nonsym", I=I, seed=I + n)
    d = upload(api, p, False)
    monkeypatch.delenv("IRS_TVLQR_VARIANT", raising=False)
    dev = api.dev
    K, k = dev.empty((I, T, m, n)), dev.empty((I, T, m))
    status = dev.empty((I,), api.torch.int32)
    api.lib.call("irs_tvlqr_riccati", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(d["Q"]),
                 dev.ptr(d["Qd"]), dev.ptr(d["R"]), dev.ptr(d["xd"]), d["xd_stride"], I, T, dev.ptr(K), dev.ptr(k),
                 dev.ptr(status), dev.stream_ptr())
    Kn, kn = api.np(K), api.np(k)
    assert np.all(api.np(status) == 0)
    Ko, ko = oracle(p, False, I)
    assert rel_err(Kn, Ko) < 1e-9 and rel_err(kn, ko) < 1e-9
    Kb, kb, sb, _, _ = riccati(api, d, n, m, I, T, "block", False, monkeypatch)
    assert rel_err(Kn, api.np(Kb)) < 1e-10 and rel_err(kn, api.np(kb)) < 1e-10


# ------------------------------------------------------------------------------------------------
# segments of the tiled kernel
# ------------------------------------------------------------------------------------------------
SPLITS = {1: [(0, 1)], 2: [(1, 2), (0, 1)], 7: [(6, 7), (2, 6), (1, 2), (0, 1)],
          100: [(99, 100), (60, 99), (59, 60), (1, 59), (0, 1)]}


@pytest.mark.parametrize("T", HORIZONS)
@pytest.mark.parametrize("n,m", [(6, 2), (12, 4)])
def test_segment_chains_are_bit_identical_to_the_full_pass(api, n, m, T, monkeypatch):
    """Uneven splits, segments of one step at both ends, T = 1: the chained segments with the carried (P, p)
    reproduce the one-launch pass bit for bit, for non-symmetric weights too."""
    I = 3
    p = problem(n, m, T, "nonsym", I=I, seed=T + n)
    d = upload(api, p, False)
    K0, k0, st0, _, _ = riccati(api, d, n, m, I, T, "block", False, monkeypatch)
    dev, torch = api.dev, api.torch
    K, k = torch.full_like(K0, float("nan")), torch.full_like(k0, float("nan"))
    st = torch.full_like(st0, -1)
    carry = dev.empty((I, n * n + n))
    for lo, hi in SPLITS[T]:
        api.lib.call("irs_tvlqr_riccati_segment", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]),
                     dev.ptr(d["Q"]), dev.ptr(d["Qd"]), dev.ptr(d["R"]), dev.ptr(d["xd"]), d["xd_stride"], I, T, lo, hi,
                     dev.ptr(carry), dev.ptr(K), dev.ptr(k), dev.ptr(st), dev.stream_ptr())
    assert torch.equal(K, K0) and torch.equal(k, k0) and torch.equal(st, st0)
    assert int(st.abs().sum().item()) == 0
    Ko, ko = oracle(p, False, I)
    assert rel_err(api.np(K), Ko) < 1e-9 and rel_err(api.np(k), ko) < 1e-9


# ------------------------------------------------------------------------------------------------
# irs_tvlqr_riccati_ex: H^-1 and P of every step
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["diag", "dense", "nonsym"])
@pytest.mark.parametrize("env", ["block", "warp"])
@pytest.mark.parametrize("n,m", DIMS)
def test_ex_outputs_match_the_oracle_hessians(api, n, m, env, kind, monkeypatch):
    """Hinv[t] = inv(sym(R)/2 + B' P_{t+1} B) and P[t] = the oracle's value-function Hessian, P[T] = sym(Qd)."""
    T, I = 7, 5
    p = problem(n, m, T, kind, I=I, seed=n + m)
    d = upload(api, p, False)
    K, k, status, Hinv, P = riccati(api, d, n, m, I, T, env, True, monkeypatch)
    assert np.all(api.np(status) == 0)
    Ko, ko, Po, Ho = oracle(p, False, I, hessians=True)
    Q, Qd, R = p["ref"]
    Hinv_o = np.linalg.inv(Ho)
    assert rel_err(api.np(Hinv), Hinv_o) < 1e-10
    assert rel_err(api.np(P), Po) < 1e-10
    Pn = api.np(P)
    assert np.array_equal(Pn[:, T], np.broadcast_to(0.5 * (Qd + Qd.T), (I, n, n)))
    assert rel_err(api.np(K), Ko) < 1e-9 and rel_err(api.np(k), ko) < 1e-9


# ------------------------------------------------------------------------------------------------
# status: one bad instance is flagged, and only it
# ------------------------------------------------------------------------------------------------
def _status_cases(n, m):
    """(label, env, ex, I, poisoned instances): warp blocks of 4 (an instance of the partial block), packed
    pairs (both halves of a warp) and the last, partial block of 8."""
    out = []
    for label, env, ex, _ in variants(n, m):
        if label == "packed":
            out.append((label, env, ex, 17, (4, 5, 16)))
        elif label == "generic-warp":
            out.append((label, env, ex, 5, (1, 4)))
        else:
            out.append((label, env, ex, 3, (1,)))
    return out


@pytest.mark.parametrize("bad", ["nan", "inf"])
@pytest.mark.parametrize("n,m", DIMS)
def test_status_flags_exactly_the_instance_with_a_bad_operand(api, n, m, bad, monkeypatch):
    """A NaN or Inf in A_t, B_t, c_t or xd_t of one instance at an interior step t: every variant sets the
    status of that instance and of no other.  (A NaN in c_t or xd_t leaves P finite and reaches k only.)"""
    T, t = 7, 3
    value = np.nan if bad == "nan" else np.inf
    base = problem(n, m, T, "dense", I=17, seed=5)
    for label, env, ex, I, victims in _status_cases(n, m):
        for field, index in (("At", (t, 0, 0)), ("Bt", (t, n - 1, 0)), ("ct", (t, 0)), ("xd", (t, 0))):
            for i in victims:
                p = dict(base)
                p[field] = base[field].copy()
                p[field][(i,) + index] = value
                d = upload(api, p, False)
                _, _, status, _, _ = riccati(api, d, n, m, I, T, env, ex, monkeypatch)
                expect = np.zeros(I, dtype=np.int32)
                expect[i] = 1
                assert np.array_equal(api.np(status), expect), (label, field, i, api.np(status))


@pytest.mark.parametrize("n,m", DIMS)
def test_status_flags_every_instance_of_a_non_spd_problem(api, n, m, monkeypatch):
    """An indefinite terminal weight fails at the first step; a negative definite Q with a positive Qd fails
    only in the middle of the horizon.  Both: every instance flagged, by every variant."""
    T = 7
    p = problem(n, m, T, "dense", I=17, seed=9)
    d = upload(api, p, False)
    cases = {"negative Qd": (p["Q"], -np.eye(n), 1e-6 * np.eye(m)),
             "negative Q": (-100.0 * np.eye(n), np.eye(n), 1e-3 * np.eye(m))}
    Q, Qd, R = cases["negative Q"]
    with pytest.raises(np.linalg.LinAlgError):
        cr.tvlqr_riccati(p["At"][0], p["Bt"][0], p["ct"][0], Q, Qd, R, p["xd"][0])
    cr.tvlqr_riccati(p["At"][0][T - 1:], p["Bt"][0][T - 1:], p["ct"][0][T - 1:], Q, Qd, R, p["xd"][0][T - 1:])
    for name, (Q, Qd, R) in cases.items():
        for label, env, ex, _ in variants(n, m):
            I = 17 if label == "packed" else 5
            _, _, status, _, _ = riccati(api, d, n, m, I, T, env, ex, monkeypatch, api.up(Q), api.up(Qd), api.up(R))
            assert np.all(api.np(status) == 1), (name, label)


# ------------------------------------------------------------------------------------------------
# irs_evaluate_cost
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T", [1, 31, 32, 33, 65])
@pytest.mark.parametrize("I", [1, 5])
@pytest.mark.parametrize("n,m", DIMS)
def test_evaluate_cost_matches_the_oracle(api, n, m, I, T):
    """Lanes run over t (32 per pass): horizons around one and two passes; a non-symmetric Q."""
    rng = np.random.default_rng(T + I)
    x = rng.standard_normal((I, T + 1, n))
    u = rng.standard_normal((I, T, m))
    xd = rng.standard_normal((I, T + 1, n))
    Q = spd(rng, n) + 0.5 * rng.standard_normal((n, n))
    R = spd(rng, m)
    dev = api.dev
    for shared in (False, True):
        dxd = api.up(xd[:1] if shared else xd)
        cost = dev.empty((I,))
        dx, du, dQ, dR = api.up(x), api.up(u), api.up(Q), api.up(R)
        api.lib.call("irs_evaluate_cost", n, m, dev.ptr(dx), dev.ptr(du), dev.ptr(dxd), 0 if shared else (T + 1) * n,
                     dev.ptr(dQ), dev.ptr(dR), I, T, dev.ptr(cost), dev.stream_ptr())
        got = api.np(cost)
        for i in range(I):
            want = cr.evaluate_cost(x[i], u[i], xd[0 if shared else i], Q, R)
            assert abs(got[i] - want) <= 1e-12 * abs(want), (i, shared, got[i], want)


# ------------------------------------------------------------------------------------------------
# the plan check: may local_descent skip the box QPs?
# ------------------------------------------------------------------------------------------------
def plans(At, Bt, ct, K, k, x_trj):
    """Every plan of plan_check_kernel restated: from x_trj[i, t0], x <- A x + B (K x + k) + c up to T.
    Returns (values [I, T, T, n + m] with NaN before t0: x_{t+1} | u_t of the plan from t0, the same in the
    kernel's order ((A + B K) x + (B k + c)))."""
    I, T, n = At.shape[0], At.shape[1], At.shape[2]
    m = Bt.shape[3]
    direct = np.full((I, T, T, n + m), np.nan)
    rows = np.full((I, T, T, n + m), np.nan)
    Acl = At + np.einsum("itnj,itjk->itnk", Bt, K)
    acl = np.einsum("itnj,itj->itn", Bt, k) + ct
    for t0 in range(T):
        x = x_trj[:, t0].copy()
        xr = x.copy()
        for t in range(t0, T):
            u = np.einsum("imn,in->im", K[:, t], x) + k[:, t]
            x = np.einsum("inj,ij->in", At[:, t], x) + np.einsum("inj,ij->in", Bt[:, t], u) + ct[:, t]
            ur = np.einsum("imn,in->im", K[:, t], xr) + k[:, t]
            xr = np.einsum("inj,ij->in", Acl[:, t], xr) + acl[:, t]
            direct[:, t0, t] = np.concatenate((x, u), axis=1)
            rows[:, t0, t] = np.concatenate((xr, ur), axis=1)
    return direct, rows


def flags(values, lo, hi, tol):
    bad = (values < lo - tol) | (values > hi + tol)      # NaN (steps before t0) compares False
    return np.any(bad.reshape(values.shape[0], -1), axis=1).astype(np.int32)


@pytest.mark.parametrize("T", [1, 2, 40])
@pytest.mark.parametrize("I", [1, 3, 37])
@pytest.mark.parametrize("n,m", DIMS)
def test_plan_check_decides_like_numpy(api, n, m, I, T):
    """Start from a box that holds every plan; for every coordinate and side, move that bound so that one
    chosen instance's plan crosses it by 1e-6 (flagged: that instance only), then so that the plan lies
    0.5 tol outside (inside the tolerance: nothing flagged).  The flags must equal numpy's with the rows
    computed by the check itself and with irs_tvlqr_plan_rows run first."""
    rng = np.random.default_rng(I * 100 + T + n)
    At = 0.9 * np.eye(n) + 0.05 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    K = 0.1 * rng.standard_normal((I, T, m, n))
    k = 0.1 * rng.standard_normal((I, T, m))
    x_trj = rng.standard_normal((I, T + 1, n))
    tol = api.BOUND_TOL
    values, values_rows = plans(At, Bt, ct, K, k, x_trj)
    # round-off of the two evaluation orders; every constructed margin is >= 1e4 times it
    roundoff = max(float(np.nanmax(np.abs(values - values_rows))), EPS * float(np.nanmax(np.abs(values))))
    assert 0.5 * tol >= 1e4 * roundoff, roundoff
    vmax = np.nanmax(values, axis=(1, 2))      # [I, n + m]
    vmin = np.nanmin(values, axis=(1, 2))
    lo0, hi0 = vmin.min(axis=0) - 1.0, vmax.max(axis=0) + 1.0
    dev = api.dev
    d = {name: api.up(v) for name, v in (("At", At), ("Bt", Bt), ("ct", ct), ("K", K), ("k", k), ("x", x_trj))}
    scratch = dev.empty((I, T, n + m, n + 1))
    violated = dev.empty((I,), api.torch.int32)
    api.lib.call("irs_tvlqr_plan_rows", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(d["K"]),
                 dev.ptr(d["k"]), I, T, dev.ptr(scratch), dev.stream_ptr())

    def check(lo, hi, rows_ready):
        dlo, dhi = api.up(lo), api.up(hi)
        api.lib.call("irs_tvlqr_plan_check", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(d["K"]),
                     dev.ptr(d["k"]), dev.ptr(d["x"]), dev.ptr(dlo[:n]), dev.ptr(dhi[:n]), dev.ptr(dlo[n:]),
                     dev.ptr(dhi[n:]), tol, I, T, rows_ready, dev.ptr(violated), dev.ptr(scratch), dev.stream_ptr())
        return api.np(violated)

    for rows_ready in (1, 0):
        assert np.array_equal(check(lo0, hi0, rows_ready), np.zeros(I, np.int32))
    for c in range(n + m):
        for side in ("lo", "hi"):
            ext = vmin[:, c] if side == "lo" else vmax[:, c]
            i = int(np.argmin(ext) if side == "lo" else np.argmax(ext))
            sign = -1.0 if side == "lo" else 1.0
            for outside, expect_i in ((tol + 1e-6, 1), (0.5 * tol, 0)):
                lo, hi = lo0.copy(), hi0.copy()
                (lo if side == "lo" else hi)[c] = ext[i] - sign * outside
                want = flags(values, lo, hi, tol)
                expect = np.zeros(I, np.int32)
                expect[i] = expect_i
                assert np.array_equal(want, expect), (c, side, outside)      # the construction itself
                # every plan value is >= 1e4 round-off away from its threshold
                thr = (lo[c] - tol) if side == "lo" else (hi[c] + tol)
                assert float(np.nanmin(np.abs(values[..., c] - thr))) >= 1e4 * roundoff
                for rows_ready in (1, 0):
                    assert np.array_equal(check(lo, hi, rows_ready), want), (c, side, outside, rows_ready)
