"""CPU: the partial-Gram reference (oracle/sample_gram.py) and the proof that the tolerances of the GPU
partial tests (tests/test_smoothing_kernels.py) have teeth.  For every system, at a chunk boundary, one sample
past it and at an odd N, and for the chunk sizes the GPU tests run (256, 1024, 1536 for the learned dynamics,
4096 = the default plan), the CPU models of both Gram engines pass their tolerance, and every kernel-bug mutation
exceeds the CUDA-core tolerance at least 10x and the tensor-core tolerance by TEETH_TC[S]: 10x up to S = 1536,
5x at S = 4096.  A bug that touches one sample shrinks like 1/S while the tensor-core floor (one bf16x2 product,
2^-16) does not; at S = 4096 the weakest mutations are a dropped sample of pendulum (1.05e-4) and the hi piece
only (1.6e-4) against 2e-5."""
import numpy as np
import pytest

from oracle import cpu_restatement as cr
from oracle import example_configs as ec
from oracle import philox_ref
from oracle import sample_gram as sg

CHUNKS = [256, 1024, 1536, 4096]                 # samples per chunk
TEETH_CC = 10.0
TEETH_TC = {256: 10.0, 1024: 10.0, 1536: 10.0, 4096: 5.0}
DIMS = {"pendulum": (2, 1), "bicycle": (5, 2), "quadrotor": (12, 4), "three_cart": (6, 2)}


def _setup(name, N, projection=None, antithetic=False):
    """Rows of nominal point t = 3 of the `_nominal` trajectory of test_gpu_parity.py, responses from the
    float64 oracle rounded to float32."""
    cfg = ec.CONFIGS[name](T=6)
    orc = cr.SYSTEMS[name](cfg["h"])
    n = orc.dim_x
    rng = np.random.default_rng(42)
    u_trj = cfg["u_trj_initial"] + 0.05 * rng.standard_normal(cfg["u_trj_initial"].shape)
    x_trj = cr.rollout(orc, cfg["x0"], u_trj)
    t = 3
    z = philox_ref.deltas(1, N, cfg["sigma"] / 3 ** cfg["power"], 99, 3, t0=t, antithetic=antithetic)[0].astype(np.float32)

    def project(xp):
        return orc.projection(xp, np.zeros_like(xp), np.zeros((xp.shape[0], 2)), np.zeros((xp.shape[0], 2)))[0]

    w, pts, (xf, uf), centred = sg.perturbed_points(x_trj[t], u_trj[t], z, projection, project)
    pts64 = pts.astype(np.float64)
    f = orc.dynamics_batch(pts64[:, :n], pts64[:, n:]).astype(np.float32)
    fr = orc.dynamics_batch if centred else orc.dynamics_scalar_batch if name == "three_cart" else orc.dynamics_batch
    fbar = fr(xf[None].astype(np.float64), uf[None].astype(np.float64))[0].astype(np.float32)
    return w, f, fbar, centred


def _moments(name, centred):
    return None if name != "three_cart" else bool(centred)


@pytest.mark.parametrize("name", list(DIMS))
def test_packed_layout_round_trips(name):
    n, m = DIMS[name]
    d, W = n + m, 2 * n + m
    G = np.arange(d * W, dtype=np.float64).reshape(d, W)
    packed = sg.pack(G, d, W)
    assert packed.shape[0] + (2 * n + m if name == "three_cart" else 0) == sg.gram_width(n, m, name == "three_cart")
    for i in range(d):
        for j in range(i, W):
            assert packed[sg.gram_row_offset(i, W) + j - i] == G[i, j]


def test_layout_matches_the_library(built_lib):
    """The packed width agrees with the CUDA library's own (irs_partial_width)."""
    for sid, name in enumerate(["pendulum", "bicycle", "quadrotor", "three_cart"]):
        n, m = DIMS[name]
        assert built_lib.irs_partial_width(sid, 0) == sg.gram_width(n, m, name == "three_cart")


CASES = [(name, k, proj) for name in DIMS for k in (0, 1, 2) for proj in (None,)] + \
        [("three_cart", k, proj) for k in (1, 2) for proj in ("delta", "absolute")]


def _n_of(S, k):
    """k = 0: N at a chunk boundary, 1: one past it, 2: odd, over two chunks."""
    return (S, S + 1, 2 * S + 1)[k]


def _bar(S):
    return max(TEETH_CC * sg.TOL_CUDA_CORES, TEETH_TC[S] * sg.TOL_TENSOR_CORES)


@pytest.mark.parametrize("S", CHUNKS)
@pytest.mark.parametrize("name,k,projection", CASES)
def test_models_pass_and_every_mutation_fails_by_10x(name, k, projection, S):
    N = _n_of(S, k)
    w, f, fbar, centred = _setup(name, N, projection)
    d = w.shape[1]
    C = (N + S - 1) // S
    rows = sg.sample_rows(w, f, fbar)
    mom = _moments(name, centred)
    ref, absref = sg.chunk_partials(rows, N, C, S, d, moments=mom)
    nacc = ref.shape[1] - (0 if mom is None else rows.shape[1])
    err_ffma = sg.normalized_error(sg.ffma_model(rows, N, C, S, d), ref[:, :nacc], absref[:, :nacc])
    err_tc = sg.normalized_error(sg.tc_model(rows, N, C, S, d), ref[:, :nacc], absref[:, :nacc])
    assert err_ffma < sg.TOL_CUDA_CORES, err_ffma
    assert err_tc < sg.TOL_TENSOR_CORES, err_tc
    bar = _bar(S)
    muts = dict(sg.ROW_MUTATIONS)
    if mom:
        muts["moment off by one sample"] = sg.mutate_moment_off_by_one
    for label, fn in muts.items():
        e = sg.normalized_error(fn(rows, N, C, S, d, moments=mom), ref, absref)
        assert e > bar, (label, e)


@pytest.mark.parametrize("S", CHUNKS)
@pytest.mark.parametrize("name", ["pendulum", "bicycle", "quadrotor"])
@pytest.mark.parametrize("k", [0, 1, 2])
def test_paired_rows_models_pass_and_mutations_fail_by_10x(name, k, S):
    """Antithetic pairs as the tensor-core kernel stages them: one row per pair, the regressor block doubled,
    a lone + member at odd N.  The paired Gram equals the per-sample Gram of the same samples up to the
    rounding of the responses."""
    N = _n_of(S, k)
    w, f, fbar, _ = _setup(name, N, antithetic=True)
    d = w.shape[1]
    C = (N + S - 1) // S
    rows = sg.paired_rows(w, f, fbar)
    ref, absref = sg.chunk_partials(rows, N, C, S, d, paired=True)
    per_sample = sg.chunk_partials(sg.sample_rows(w, f, fbar), N, C, S, d)
    assert sg.normalized_error(per_sample[0], ref, absref) < 1e-5
    err_tc = sg.normalized_error(sg.tc_model(rows, N, C, S, d, paired=True), ref, absref)
    assert err_tc < sg.TOL_TENSOR_CORES, err_tc
    bar = _bar(S)
    for label, fn in sg.ROW_MUTATIONS.items():
        e = sg.normalized_error(fn(rows, N, C, S, d, paired=True), ref, absref)
        assert e > bar, (label, e)
    for label, fn in sg.PAIR_MUTATIONS.items():
        if label == "lone member unscaled" and N % 2 == 0:
            continue
        e = sg.normalized_error(fn(w, f, fbar, N, C, S, d), ref, absref)
        assert e > bar, (label, e)


def test_normalized_error_demands_exact_zeros_and_rejects_nan():
    ref = np.array([[0.0, 1.0]])
    absref = np.array([[0.0, 1.0]])
    assert sg.normalized_error(np.array([[0.0, 1.0]]), ref, absref) == 0.0
    assert sg.normalized_error(np.array([[1e-30, 1.0]]), ref, absref) == np.inf
    assert sg.normalized_error(np.array([[0.0, np.nan]]), ref, absref) == np.inf
