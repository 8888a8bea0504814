"""TVLQR at state and input dimensions chosen at run time (csrc/tvlqr_any.cuh), through the C ABI and `solve_tvlqr`.

The kernels of csrc/tvlqr.cuh and csrc/tvlqr_box.cuh are instantiated for the built-in pairs (2,1), (5,2), (6,2)
and (12,4) only; `irs_tvlqr_riccati_any`, `irs_tvlqr_linear_rollout_any` and `irs_tvlqr_box_qp_any` take any
1 <= n, m <= 32, the built-in pairs included, and are pinned here to the same references and bars as the built-in
kernels (tests/test_lqr_kernels.py, tests/test_box_qp_kernels.py):

- gains against the recursion oracle `cr.tvlqr_riccati` (1e-9, or 1e-15 cond(H) for ill-conditioned weights);
  H^-1 and P against the oracle's (1e-10); u* of the linear rollout against the dense KKT solve
  `oracle/dense_lqr.py`; at the built-in pairs the gains against the templated kernels (1e-10);
- box QPs against the exact KKT certificate of `oracle/box_kkt.py` (1e-7 max(1, |.*|_inf)) and the numpy ADMM
  `oracle/box_tvlqr.py` (1e-7);
- `solve_tvlqr` on a cart-pole (n = 4, m = 1) linearized by central differences, bounded and unbounded.

The CPU tests check the host-side validation, which runs before any launch.
"""
import ctypes

import numpy as np
import pytest

from oracle import box_kkt as bk
from oracle import box_tvlqr as bq
from oracle import cpu_restatement as cr
from oracle import dense_lqr

BUILTIN = [(2, 1), (5, 2), (6, 2), (12, 4)]
NEW_DIMS = [(1, 1), (3, 1), (4, 1), (3, 3), (6, 3), (7, 5), (16, 8), (31, 2), (32, 32)]
HORIZONS = [1, 2, 7, 100]
WEIGHTS = ["diag", "dense", "nonsym", "illcond", "scale+30", "scale-30"]
COUNTS = (1, 3, 17)
I_MAX = 17
BAR = 1e-7
SMEM_LIMIT = 200 * 1024


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-300))


def box_smem_bytes(n, m, T, cache):
    """box_qp_any_smem_bytes of csrc/tvlqr_any.cuh, restated: keep the two in step."""
    d = 3 * (T + 1) * n + 4 * T * m + T * n + (T + 1) * n + 2 * n + n + m
    if cache:
        d += T * (n * n + 2 * n * m + m * m + n)
    return 8 * d


def t_cache(n, m):
    return max(T for T in range(1, 4000) if box_smem_bytes(n, m, T, True) <= SMEM_LIMIT)


def t_max(n, m):
    return max(T for T in range(1, 4000) if box_smem_bytes(n, m, T, False) <= SMEM_LIMIT)


# ------------------------------------------------------------------------------------------------
# CPU: limits and host-side validation
# ------------------------------------------------------------------------------------------------
def test_limits(built_lib):
    a, b = ctypes.c_int(), ctypes.c_int()
    assert built_lib.irs_tvlqr_any_limits(ctypes.byref(a), ctypes.byref(b)) == 0
    assert (a.value, b.value) == (32, 32)
    assert built_lib.irs_tvlqr_any_limits(None, ctypes.byref(b)) != 0
    assert b"null pointer" in built_lib.irs_last_error()
    from irs_mpc_b200 import tv_lqr
    assert tv_lqr.tvlqr_any_limits() == (32, 32)


def test_box_layout_boundaries():
    assert (t_cache(32, 32), t_max(32, 32)) == (5, 88)
    assert (t_cache(4, 1), t_max(4, 1)) == (482, 1065)


def _riccati_any(lib, n, m, I=1, T=1, ptr=1, xd_stride=0):
    return lib.irs_tvlqr_riccati_any(n, m, ptr, 1, 1, 1, 1, 1, 1, xd_stride, I, T, 1, 1, 1, None, None, None)


def _rollout_any(lib, n, m, I=1, T=1, ptr=1):
    return lib.irs_tvlqr_linear_rollout_any(n, m, ptr, 1, 1, 1, 1, 1, I, T, 1, 1, None)


def _box_any(lib, n, m, I=1, T=1, ptr=1, xs=0, us=0, alpha=1.6, max_iter=10):
    return lib.irs_tvlqr_box_qp_any(n, m, ptr, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, 1, xs, us, 1,
                                    alpha, 1e-10, max_iter, I, T, 1, 1, 1, 1, None)


@pytest.mark.parametrize("entry", [_riccati_any, _rollout_any, _box_any])
def test_validation_messages(built_lib, entry):
    """Every argument error is returned before a launch, so without a GPU too."""
    lib = built_lib
    for n, m in ((0, 1), (33, 1), (1, 0), (4, 33), (-1, -1)):
        assert entry(lib, n, m) != 0
        assert b"out of range" in lib.irs_last_error(), (n, m)
    assert entry(lib, 4, 1, ptr=None) != 0 and b"null pointer" in lib.irs_last_error()
    assert entry(lib, 4, 1, I=0) != 0 and b"I >= 1" in lib.irs_last_error()
    assert entry(lib, 4, 1, T=0) != 0 and b"T >= 1" in lib.irs_last_error()


def test_validation_of_the_box_qp(built_lib):
    lib = built_lib
    for xs, us in ((1, 0), (0, 2), (5, 1), (4, 3)):
        assert _box_any(lib, 4, 1, xs=xs, us=us) != 0
        assert b"box strides" in lib.irs_last_error(), (xs, us)
    assert _box_any(lib, 4, 1, alpha=2.0) != 0 and b"alpha" in lib.irs_last_error()
    assert _box_any(lib, 4, 1, max_iter=0) != 0 and b"max_iter" in lib.irs_last_error()
    assert _box_any(lib, 32, 32, T=89) != 0
    msg = lib.irs_last_error()
    assert b"T=89 too long" in msg and b"longest is T=88" in msg, msg
    assert _riccati_any(lib, 4, 1, xd_stride=-1) != 0 and b"xd_stride" in lib.irs_last_error()


def test_the_built_in_entry_points_keep_their_dims(built_lib):
    from irs_mpc_b200 import tv_lqr
    assert built_lib.irs_tvlqr_riccati(3, 3, 1, 1, 1, 1, 1, 1, 1, 0, 1, 1, 1, 1, 1, None) != 0
    assert b"unsupported TVLQR dims" in built_lib.irs_last_error()
    with pytest.raises(NotImplementedError):
        tv_lqr._DimsOnlySystem(4, 1)
    assert all(tv_lqr._builtin_dims(n, m) for n, m in BUILTIN)
    assert not any(tv_lqr._builtin_dims(n, m) for n, m in NEW_DIMS)


@pytest.mark.parametrize("n,m", [(33, 1), (1, 33), (40, 40)])
def test_solve_tvlqr_beyond_the_limits_raises(built_lib, n, m):
    """Refused before anything reaches a device."""
    from irs_mpc_b200.tv_lqr import solve_tvlqr
    T = 3
    with pytest.raises(NotImplementedError, match="n=%d states and m=%d inputs" % (n, m)):
        solve_tvlqr(np.zeros((T, n, n)), np.zeros((T, n, m)), np.zeros((T, n)), np.eye(n), np.eye(n), np.eye(m),
                    np.zeros(n), np.zeros((T + 1, n)))


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
class Api:
    def __init__(self):
        import torch
        import irs_mpc_b200.all as mod
        from irs_mpc_b200 import _device, _lib, tv_lqr
        self.torch, self.dev, self.lib, self.tv, self.m = torch, _device, _lib, tv_lqr, mod

    def up(self, a):
        return self.dev.to_device(np.ascontiguousarray(a, dtype=np.float64))

    def np(self, t):
        return self.dev.to_numpy(t)


@pytest.fixture(scope="module")
def api():
    import torch
    assert torch.cuda.is_available()
    return Api()


def spd(rng, d, lo=0.5):
    M = rng.standard_normal((d, d))
    return M.dot(M.T) / d + lo * np.eye(d)


def problem(n, m, T, kind, I=I_MAX, seed=0):
    """The random affine problems and weight kinds of tests/test_lqr_kernels.py."""
    rng = np.random.default_rng(seed)
    At = np.eye(n) + 0.1 * rng.standard_normal((I, T, n, n))
    Bt = 0.3 * rng.standard_normal((I, T, n, m))
    ct = 0.1 * rng.standard_normal((I, T, n))
    xd = rng.standard_normal((I, T + 1, n))
    x0 = rng.standard_normal((I, n))
    if kind == "diag":
        Q, Qd, R = np.diag(rng.uniform(0.5, 2, n)), np.diag(rng.uniform(5, 20, n)), np.diag(rng.uniform(0.5, 2, m))
    elif kind == "illcond":
        Q = np.diag(rng.permutation(np.logspace(-4, 4, n)))
        Qd = np.diag(rng.permutation(np.logspace(-4, 4, n)))
        R = 1e-8 * np.diag(np.logspace(0, 4, m))
        Bt = Bt * np.logspace(0, -3, m)
    else:
        Q, Qd, R = spd(rng, n), 10 * spd(rng, n), spd(rng, m)
        if kind == "nonsym":
            Q, Qd, R = (W + (lambda S: S - S.T)(rng.standard_normal(W.shape)) for W in (Q, Qd, R))
    ref = (Q, Qd, R)
    if kind.startswith("scale"):
        s = 10.0 ** int(kind[5:])
        Q, Qd, R = s * Q, s * Qd, s * R
    return dict(At=At, Bt=Bt, ct=ct, Q=Q, Qd=Qd, R=R, xd=xd, x0=x0, ref=ref, n=n, m=m, T=T)


def upload(api, p, shared):
    d = {k: api.up(p[k]) for k in ("At", "Bt", "ct", "Q", "Qd", "R", "x0")}
    d["xd"] = api.up(p["xd"][:1] if shared else p["xd"])
    d["xd_stride"] = 0 if shared else (p["T"] + 1) * p["n"]
    return d


def riccati_any(api, d, n, m, I, T, hessians=False, Q=None, Qd=None, R=None):
    """irs_tvlqr_riccati_any on the first I instances -> numpy (K, k, status, Hinv, P); outputs NaN-filled first."""
    dev, torch = api.dev, api.torch
    K = torch.full((I, T, m, n), float("nan"), dtype=torch.float64, device="cuda")
    k = torch.full((I, T, m), float("nan"), dtype=torch.float64, device="cuda")
    status = torch.full((I,), -1, dtype=torch.int32, device="cuda")
    Hinv = torch.full((I, T, m, m), float("nan"), dtype=torch.float64, device="cuda") if hessians else None
    P = torch.full((I, T + 1, n, n), float("nan"), dtype=torch.float64, device="cuda") if hessians else None
    Q, Qd, R = (d[key] if v is None else v for key, v in (("Q", Q), ("Qd", Qd), ("R", R)))
    api.lib.call("irs_tvlqr_riccati_any", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(Q),
                 dev.ptr(Qd), dev.ptr(R), dev.ptr(d["xd"]), d["xd_stride"], I, T, dev.ptr(K), dev.ptr(k),
                 dev.ptr(status), dev.ptr(Hinv) if hessians else None, dev.ptr(P) if hessians else None,
                 dev.stream_ptr())
    torch.cuda.synchronize()
    out = [api.np(K), api.np(k), api.np(status)]
    return out + ([api.np(Hinv), api.np(P)] if hessians else [None, None])


def rollout_any(api, d, n, m, I, T, K, k):
    dev = api.dev
    xs, us = dev.empty((I, T + 1, n)), dev.empty((I, T, m))
    dK, dk = api.up(K), api.up(k)      # held until the launch: a freed block can be handed to the next upload
    api.lib.call("irs_tvlqr_linear_rollout_any", n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]),
                 dev.ptr(dK), dev.ptr(dk), dev.ptr(d["x0"]), I, T, dev.ptr(xs), dev.ptr(us), dev.stream_ptr())
    return api.np(xs), api.np(us)


def oracle(p, shared, I, hessians=False):
    Q, Qd, R = p["ref"]
    xd = p["xd"][:1] if shared else p["xd"]
    out = [cr.tvlqr_riccati(p["At"][i], p["Bt"][i], p["ct"][i], Q, Qd, R, xd[0 if shared else i],
                            return_hessians=hessians) for i in range(I)]
    return [np.stack([o[j] for o in out]) for j in range(len(out[0]))]


def tolerances(p, kind, H):
    """(against the oracle / the dense QP, against the templated kernels): those of tests/test_lqr_kernels.py."""
    if kind != "illcond":
        return 1e-9, 1e-10
    cond = max(float(np.linalg.cond(h)) for h in H.reshape(-1, p["m"], p["m"]))
    return max(1e-9, 1e-15 * cond), max(1e-10, 1e-16 * cond)


def templated(api, d, n, m, I, T, hessians=False):
    """The built-in kernels at a built-in pair: irs_tvlqr_riccati (default dispatch) or irs_tvlqr_riccati_ex."""
    dev = api.dev
    K, k = dev.empty((I, T, m, n)), dev.empty((I, T, m))
    status = dev.empty((I,), api.torch.int32)
    head = (n, m, dev.ptr(d["At"]), dev.ptr(d["Bt"]), dev.ptr(d["ct"]), dev.ptr(d["Q"]), dev.ptr(d["Qd"]),
            dev.ptr(d["R"]), dev.ptr(d["xd"]), d["xd_stride"], I, T, dev.ptr(K), dev.ptr(k), dev.ptr(status))
    if hessians:
        Hinv, P = dev.empty((I, T, m, m)), dev.empty((I, T + 1, n, n))
        api.lib.call("irs_tvlqr_riccati_ex", *head, dev.ptr(Hinv), dev.ptr(P), dev.stream_ptr())
        return api.np(K), api.np(k), api.np(status), api.np(Hinv), api.np(P)
    api.lib.call("irs_tvlqr_riccati", *head, dev.stream_ptr())
    return api.np(K), api.np(k), api.np(status), None, None


# ------------------------------------------------------------------------------------------------
# GPU: Riccati and rollout
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", WEIGHTS)
@pytest.mark.parametrize("T", HORIZONS)
@pytest.mark.parametrize("n,m", NEW_DIMS + BUILTIN)
def test_gains_and_rollout_match_the_oracle_and_the_dense_qp(api, n, m, T, kind):
    p = problem(n, m, T, kind, seed=1000 * n + 100 * m + T + WEIGHTS.index(kind))
    Q, Qd, R = p["ref"]
    for shared in (False, True):
        d = upload(api, p, shared)
        Ko, ko, _, Ho = oracle(p, shared, I_MAX, hessians=True)
        tol, tol_x = tolerances(p, kind, Ho)
        for I in COUNTS:
            K, k, status, _, _ = riccati_any(api, d, n, m, I, T)
            where = (I, "shared xd" if shared else "xd per instance")
            assert np.all(status == 0), where + (status,)
            assert rel_err(K, Ko[:I]) < tol and rel_err(k, ko[:I]) < tol, where + (rel_err(K, Ko[:I]), rel_err(k, ko[:I]))
            if (n, m) in BUILTIN:
                Kt, kt, st, _, _ = templated(api, d, n, m, I, T)
                assert np.all(st == 0)
                assert rel_err(K, Kt) < tol_x and rel_err(k, kt) < tol_x, where + (rel_err(K, Kt), rel_err(k, kt))
        # u* of the linear model from x0 (the solve_tvlqr path) against the dense KKT solve.  The dense solve of
        # the largest systems takes seconds of CPU: there, one xd layout (the gains of both are checked above)
        if shared and T * (2 * n + m) > 3000:
            continue
        xs, us = rollout_any(api, d, n, m, I, T, K, k)
        for i in ((0,) if T > 7 else (0, I - 1)):
            xd = p["xd"][0 if shared else i]
            xo, uo = dense_lqr.solve(p["At"][i], p["Bt"][i], p["ct"][i], Q, Qd, R, p["x0"][i], xd)
            assert rel_err(us[i], uo) < tol, where + (i, rel_err(us[i], uo))
            assert rel_err(xs[i], xo) < tol, where + (i, rel_err(xs[i], xo))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["diag", "dense", "nonsym"])
@pytest.mark.parametrize("n,m", NEW_DIMS + BUILTIN)
def test_hessian_outputs_match_the_oracle(api, n, m, kind):
    """Hinv[t] = inv(sym(R)/2 + B' P_{t+1} B), P[t] = the oracle's value-function Hessian, P[T] = sym(Qd) exactly;
    at the built-in pairs also against irs_tvlqr_riccati_ex.  The gains do not depend on asking for them."""
    T, I = 7, 5
    p = problem(n, m, T, kind, I=I, seed=n + m)
    d = upload(api, p, False)
    K, k, status, Hinv, P = riccati_any(api, d, n, m, I, T, hessians=True)
    assert np.all(status == 0)
    Ko, ko, Po, Ho = oracle(p, False, I, hessians=True)
    Q, Qd, R = p["ref"]
    assert rel_err(Hinv, np.linalg.inv(Ho)) < 1e-10
    assert rel_err(P, Po) < 1e-10
    assert np.array_equal(P[:, T], np.broadcast_to(0.5 * (Qd + Qd.T), (I, n, n)))
    assert rel_err(K, Ko) < 1e-9 and rel_err(k, ko) < 1e-9
    K2, k2, _, _, _ = riccati_any(api, d, n, m, I, T)
    assert np.array_equal(K, K2) and np.array_equal(k, k2)
    if (n, m) in BUILTIN:
        _, _, st, Ht, Pt = templated(api, d, n, m, I, T, hessians=True)
        assert np.all(st == 0)
        assert rel_err(Hinv, Ht) < 1e-10 and rel_err(P, Pt) < 1e-10


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", NEW_DIMS + BUILTIN)
def test_status_flags(api, n, m):
    """A NaN in one instance's c_t or xd_t flags that instance and no other; an indefinite H (R negative
    definite, Qd tiny) flags every instance."""
    T, t, I = 7, 3, 3
    base = problem(n, m, T, "dense", I=I, seed=5)
    for field, index in (("ct", (t, 0)), ("xd", (t, n - 1))):
        for i in range(I):
            p = dict(base)
            p[field] = base[field].copy()
            p[field][(i,) + index] = np.nan
            d = upload(api, p, False)
            _, _, status, _, _ = riccati_any(api, d, n, m, I, T, hessians=(i == 1))
            expect = np.zeros(I, dtype=np.int32)
            expect[i] = 1
            assert np.array_equal(status, expect), (field, i, status)
    d = upload(api, base, False)
    _, _, status, _, _ = riccati_any(api, d, n, m, I, T, Qd=api.up(1e-6 * np.eye(n)), R=api.up(-np.eye(m)))
    assert np.all(status == 1), status


# ------------------------------------------------------------------------------------------------
# GPU: box-constrained QP
# ------------------------------------------------------------------------------------------------
BOX_DIMS = [(3, 1), (4, 1), (6, 3), (16, 8), (32, 32)]


def box_solve(api, p, max_iter=None):
    n, m, T = p["n"], p["m"], p["T"]
    d = {k: api.up(p[k]) for k in ("At", "Bt", "ct", "xd", "x0")}
    kw = {} if max_iter is None else {"max_iter": max_iter}
    out = api.tv.box_qp_any_device(d["At"], d["Bt"], d["ct"], api.up(p["Q"]), api.up(p["Qd"]), api.up(p["R"]),
                                   p["Q"], p["Qd"], p["R"], d["xd"], 0 if p["shared_xd"] else (T + 1) * n, d["x0"],
                                   p["xlo"], p["xhi"], p["ulo"], p["uhi"], **kw)
    return tuple(api.np(v) for v in out)


def check_instance(p, i, x, u, status, iters, margins=True):
    """The checks of check_instance in tests/test_box_qp_kernels.py (this entry returns no cost)."""
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
    xr = qp.states(u[i])
    assert np.max(np.abs(x[i] - xr)) <= 1e-12 * max(1.0, np.max(np.abs(xr))), where
    xs = max(1.0, np.max(np.abs(x[i])))
    us = max(1.0, np.max(np.abs(u[i])))
    assert np.all(x[i][1:] >= bk._rows(p["xlo"], p["T"], 1) - BAR * xs), where
    assert np.all(x[i][1:] <= bk._rows(p["xhi"], p["T"], 1) + BAR * xs), where
    assert np.all(u[i] >= bk._rows(p["ulo"], p["T"], 0) - BAR * us), where
    assert np.all(u[i] <= bk._rows(p["uhi"], p["T"], 0) + BAR * us), where
    return c


@pytest.mark.gpu
@pytest.mark.parametrize("box", ["input", "state", "both", "tv", "wide"])
@pytest.mark.parametrize("n,m", BOX_DIMS)
def test_box_qp_is_certified_and_matches_the_numpy_admm(api, n, m, box):
    """Three instances, the middle one deep inside the box."""
    T, I = 12, 3
    p = bk.make_problem(n, m, T, box, "dense", I=I, inactive=(1,), seed=1000 * n + 10 * m + len(box))
    x, u, status, iters = box_solve(api, p)
    n_active = 0
    for i in range(I):
        c = check_instance(p, i, x, u, status, iters)
        if box == "wide" or i == 1:
            assert not np.any(c["active"]), i
        n_active += int(np.sum(c["active"]))
        xo, uo, _ = bq.admm_box_qp(p["At"][i], p["Bt"][i], p["ct"][i], p["Q"], p["Qd"], p["R"], p["x0"][i],
                                   p["xd"][i], p["xlo"], p["xhi"], p["ulo"], p["uhi"])
        assert np.max(np.abs(u[i] - uo)) <= BAR * max(1.0, np.max(np.abs(uo))), i
        assert np.max(np.abs(x[i] - xo)) <= BAR * max(1.0, np.max(np.abs(xo))), i
    if box != "wide":
        assert n_active >= 2, n_active


@pytest.mark.gpu
@pytest.mark.parametrize("T", [t_cache(4, 1), t_cache(4, 1) + 1, t_max(4, 1)])
def test_box_qp_both_layouts(api, T):
    """(4, 1): the longest horizon with the per-step matrices in shared memory, the shortest without, and the
    longest accepted at all."""
    p = bk.make_problem(4, 1, T, "input", "dense", I=2, seed=T)
    x, u, status, iters = box_solve(api, p)
    for i in range(2):
        check_instance(p, i, x, u, status, iters, margins=False)


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(4, 1), (32, 32)])
def test_box_qp_horizon_limit(api, n, m):
    """T_max is solved (certified), T_max + 1 refused before launch with the limit in the message."""
    T = t_max(n, m)
    p = bk.make_problem(n, m, T, "input", "diag", I=1, seed=n)
    x, u, status, iters = box_solve(api, p)
    check_instance(p, 0, x, u, status, iters, margins=False)
    q = bk.make_problem(n, m, T + 1, "wide", "diag", I=1, seed=n)
    with pytest.raises(api.lib.IrsCudaError, match="T=%d too long.*longest is T=%d" % (T + 1, T)):
        box_solve(api, q)


@pytest.mark.gpu
def test_box_qp_unreachable_state_box_fails(api):
    """x_1 boxed far beyond what the boxed input can reach: status 1 after exactly max_iter iterations."""
    n, m, T = 4, 1, 6
    p = bk.make_problem(n, m, T, "input", "diag", I=1, seed=11)
    xlo, xhi = np.full((T + 1, n), -1e4), np.full((T + 1, n), 1e4)
    xlo[1, 0] = 1e3
    p["xlo"], p["xhi"] = xlo, xhi
    _, _, status, iters = box_solve(api, p, max_iter=500)
    assert status[0] == 1 and iters[0] == 500


# ------------------------------------------------------------------------------------------------
# GPU: the public path on a cart-pole
# ------------------------------------------------------------------------------------------------
def cartpole_step(x, u, h=0.02, mc=1.0, mp=0.1, l=0.5, g=9.81):
    """Cart-pole (cart position, pole angle from upright, their rates) under a horizontal force, explicit Euler."""
    _, th, dp, dth = x
    s, c = np.sin(th), np.cos(th)
    tmp = (u[0] + mp * l * dth ** 2 * s) / (mc + mp)
    ddth = (g * s - c * tmp) / (l * (4.0 / 3.0 - mp * c ** 2 / (mc + mp)))
    ddp = tmp - mp * l * ddth * c / (mc + mp)
    return x + h * np.array([dp, dth, ddp, ddth])


def cartpole_problem(T=100, eps=1e-6):
    """Linearization along a nominal trajectory (central differences), the affine offset c_t = f - A x - B u."""
    x0 = np.array([0.0, 0.4, 0.0, 0.0])
    u_nom = 0.5 * np.sin(0.1 * np.arange(T))[:, None]
    x_nom = [x0]
    for t in range(T):
        x_nom.append(cartpole_step(x_nom[-1], u_nom[t]))
    x_nom = np.array(x_nom)
    At, Bt, ct = np.zeros((T, 4, 4)), np.zeros((T, 4, 1)), np.zeros((T, 4))
    for t in range(T):
        for j in range(5):
            dz = np.zeros(5)
            dz[j] = eps
            fp = cartpole_step(x_nom[t] + dz[:4], u_nom[t] + dz[4:])
            fm = cartpole_step(x_nom[t] - dz[:4], u_nom[t] - dz[4:])
            (At[t][:, j] if j < 4 else Bt[t][:, 0])[:] = (fp - fm) / (2 * eps)
        ct[t] = cartpole_step(x_nom[t], u_nom[t]) - At[t].dot(x_nom[t]) - Bt[t].dot(u_nom[t])
    Q, Qd, R = np.diag([1.0, 10.0, 0.1, 0.1]), np.diag([100.0, 1000.0, 10.0, 10.0]), np.array([[0.1]])
    xd = np.zeros((T + 1, 4))
    return At, Bt, ct, Q, Qd, R, x0, xd


@pytest.mark.gpu
def test_solve_tvlqr_on_a_cartpole(api):
    At, Bt, ct, Q, Qd, R, x0, xd = cartpole_problem()
    T = At.shape[0]
    xs, us = api.m.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd, None)
    xo, uo = dense_lqr.solve(At, Bt, ct, Q, Qd, R, x0, xd)
    assert rel_err(us, uo) < 1e-9 and rel_err(xs, xo) < 1e-9
    # an input box the unconstrained plan leaves: the bounded QP, certified
    f = 0.5 * float(np.max(np.abs(uo)))
    ub = np.stack((np.full((T, 1), -f), np.full((T, 1), f)))
    xb = np.stack((np.full(4, -1e3), np.full(4, 1e3)))
    xs, us = api.m.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd, None, x_bound_abs=xb, u_bound_abs=ub)
    qp = bk.BoxQP(At, Bt, ct, Q, Qd, R, x0, xd, xb[0], xb[1], ub[0], ub[1])
    c = qp.certify(us)
    assert c["certified"] and np.any(c["active"])
    assert np.max(np.abs(us - c["u"])) <= BAR * max(1.0, np.max(np.abs(c["u"])))
    assert np.max(np.abs(xs - c["x"])) <= BAR * max(1.0, np.max(np.abs(c["x"])))
    assert np.max(np.abs(us)) <= f * (1 + BAR)
    # a start state outside its box: the reference's infeasible QP
    xb0 = xb.copy()
    xb0[1, 1] = 0.3
    with pytest.raises(ValueError, match="TV_LQR failed"):
        api.m.solve_tvlqr(At, Bt, ct, Q, Qd, R, x0, xd, None, x_bound_abs=xb0, u_bound_abs=ub)
