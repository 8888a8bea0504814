"""CPU reference for the per-chunk partial Gram blocks of the zero-order accumulate kernels (numpy only).

The accumulate kernels (smooth.cuh: smooth_zero_order_kernel, smooth_tc.cuh: smooth_zero_order_tc_kernel,
smooth_mlp.cuh: smooth_zero_order_mlp_kernel) write, per (nominal point p, chunk c), the packed upper rows of
    G = sum_s a_s b_s^T,   a_s = regressor row (d = n + m),   b_s = [regressors | response] (W = d + n)
over the samples [c S, min((c + 1) S, N)), followed for centred-capable systems (three_cart) by the first
moments [sum_s z'_s (d) | sum_s dF_s (n)].  Row i of the packed block holds columns j = i .. W - 1 and starts at
gram_row_offset(i, W) = i W - i (i - 1) / 2.

The fit that follows is a least-squares regression whose answer barely moves when samples are dropped,
duplicated or re-weighted, so a fit-level comparison cannot see those bugs.  They are obvious in the partials:
this module forms each sample's row exactly as the kernel forms it (in float32, from the same fp32 responses),
sums the rows in float64, and measures a kernel's block against it entry by entry in units of
sum_s |a_si| |b_sj| (`normalized_error`).  It also carries CPU models of the two Gram engines' rounding and a
set of kernel-bug mutations, so that the CPU tests can show the tolerance accepts the first and rejects the
second.
"""
import numpy as np

F32 = np.float32
# Largest normalized partial error accepted from each Gram engine (tests/test_smoothing_kernels.py).  The CPU
# models of the engines stay below them; every mutation below exceeds the CUDA-core one at least 10x, the
# tensor-core one 10x for chunks of up to 1536 samples and 5x at 4096 (tests/test_oracle_sample_gram.py).  The tensor-core split keeps 16 significant bits of every value (bf16 hi +
# bf16 lo), so one product can be off by 2^-16 = 1.5e-5 relative: a chunk of a single sample reaches that.
# That leaves the tensor-core tolerance little room: the largest error of the GPU tests on a B200 was 1.42e-5
# (1.4x below it), the worst single bf16x2 product about 1.46e-5 (1.35x).  Both are deterministic for the fixed
# seeds of the tests, but another seed or configuration can come closer; 2^-16 is a floor, not noise.
TOL_CUDA_CORES = 2e-6
TOL_TENSOR_CORES = 2e-5
# the lone + member of an odd paired chunk (smooth_tc.cuh, kTcPaired): [z / sqrt 2 | sqrt 2 (f+ - fbar)]
INV_SQRT2_F32 = F32(0.70710678118654752)
SQRT2_F32 = F32(1.41421356237309505)


def gram_row_offset(i, W):
    return i * W - i * (i - 1) // 2


def gram_width(n, m, centered_capable):
    d = n + m
    return d * (d + 1) // 2 + d * n + (2 * n + m if centered_capable else 0)


# --------------------------------------------------------------------------------------------------
# sample rows
# --------------------------------------------------------------------------------------------------
def centred_frame(x_nom, u_nom):
    """systems.cuh: centred_frame for three_cart: the doubled nominal, positions and velocities relative to
    cart 1's, rounded to float32 from float64."""
    xb = np.asarray(x_nom, dtype=np.float64)
    xf = np.zeros(6, dtype=F32)
    xf[1], xf[2] = F32(2.0 * (xb[1] - xb[0])), F32(2.0 * (xb[2] - xb[0]))
    xf[4], xf[5] = F32(2.0 * (xb[4] - xb[3])), F32(2.0 * (xb[5] - xb[3]))
    return xf, (2.0 * np.asarray(u_nom, dtype=np.float64)).astype(F32)


def perturbed_points(x_nom, u_nom, z, projection=None, project=None, replay_absolute=False, proj_dims=3):
    """The regressors w [N, d] (float32) and the float32 points [N, d] the kernel evaluates the sample dynamics
    at, plus the float32 frame (x, u) the nominal response is measured at and whether the launch is centred.

    z: the float32 deltas (Philox or replayed).  projection: None | "delta" | "absolute" (three_cart's
    IRS_PROJECT_DELTA / IRS_PROJECT_ABSOLUTE); project(x [N, n] float64) -> projected absolute points, in
    float64 (the kernel projects the positions in fp64, smooth.cuh: project_deltas).  replay_absolute: z
    holds replayed ABSOLUTE points and the launch sets IRS_CENTERED (w = fl32(z - nominal) in fp64)."""
    xb = np.asarray(x_nom, dtype=np.float64)
    ub = np.asarray(u_nom, dtype=np.float64)
    n = xb.shape[0]
    w = np.array(z, dtype=F32)
    if projection is not None:
        xp = xb[None, :] + w[:, :n].astype(np.float64)
        xp = project(xp)
        w[:, :proj_dims] = (xp[:, :proj_dims] - xb[None, :proj_dims]).astype(F32)
    if replay_absolute:
        w[:, :n] = (w[:, :n].astype(np.float64) - xb[None, :]).astype(F32)
        w[:, n:] = (w[:, n:].astype(np.float64) - ub[None, :]).astype(F32)
    centred = projection == "absolute" or replay_absolute
    if centred:
        xf, uf = centred_frame(xb, ub)
    else:
        xf, uf = xb.astype(F32), ub.astype(F32)
    pts = (np.concatenate((xf, uf))[None, :] + w).astype(F32)
    return w, pts, (xf, uf), centred


def sample_rows(w, f, fbar):
    """One row per sample: [w | fl32(f - fbar)] (float32 [N, d + n])."""
    resp = (np.asarray(f, dtype=F32) - np.asarray(fbar, dtype=F32)[None, :]).astype(F32)
    return np.hstack((np.asarray(w, dtype=F32), resp))


def paired_rows(w, f, fbar):
    """Antithetic pairs on the tensor cores (smooth_tc.cuh, kTcPaired without projection): samples 2q, 2q + 1
    are x + z_q, x - z_q and stage ONE row [z_q | fl32(f+ - f-)]; the regressor block of the pair is 2 z z^T
    (chunk_partials(paired=True) doubles it).  A lone + member (odd N) stages
    [fl32(z 0.70710678f) | fl32(1.41421356f fl32(f+ - fbar))]."""
    w = np.asarray(w, dtype=F32)
    f = np.asarray(f, dtype=F32)
    N = w.shape[0]
    q = N // 2
    rows = [np.hstack((w[0:2 * q:2], (f[0:2 * q:2] - f[1:2 * q:2]).astype(F32)))]
    if N % 2:
        lone_w = (w[-1:] * INV_SQRT2_F32).astype(F32)
        lone_f = (SQRT2_F32 * (f[-1:] - np.asarray(fbar, dtype=F32)[None, :]).astype(F32)).astype(F32)
        rows.append(np.hstack((lone_w, lone_f)))
    return np.vstack(rows).astype(F32)


# --------------------------------------------------------------------------------------------------
# packed partials
# --------------------------------------------------------------------------------------------------
def pack(G, d, W):
    """[d, W] full block -> packed upper rows (the kernel's layout)."""
    return np.concatenate([G[i, i:W] for i in range(d)])


def chunk_bounds(N, C, S, paired=False):
    """Row ranges of the C chunks: samples [c S, min((c + 1) S, N)), or the pair rows of them (S is even)."""
    if paired:
        rows = (N + 1) // 2
        return [(c * S // 2, min((c + 1) * S // 2, rows)) for c in range(C)]
    return [(c * S, min((c + 1) * S, N)) for c in range(C)]


def chunk_partials(rows, N, C, S, d, paired=False, moments=None, bounds=None):
    """float64 sums and absolute sums per packed entry, [C, width] each.

    rows: float32 [R, d + n] (sample_rows or paired_rows).  moments: None (no first-moment slots), False
    (the slots exist and must be 0: a non-centred launch of a centred-capable system), True (sums of the row's
    [z' | dF] columns).  bounds: row ranges per chunk (default chunk_bounds)."""
    r = np.asarray(rows, dtype=np.float64)
    W = r.shape[1]
    n = W - d
    bounds = chunk_bounds(N, C, S, paired) if bounds is None else bounds
    nmom = 0 if moments is None else d + n
    width = d * (d + 1) // 2 + d * n + nmom
    ref = np.zeros((C, width))
    absref = np.zeros((C, width))
    scale = np.ones((d, W))
    if paired:
        scale[:, :d] = 2.0
    for c, (lo, hi) in enumerate(bounds):
        blk = r[lo:hi]
        ref[c, :width - nmom] = pack(scale * (blk[:, :d].T @ blk), d, W)
        absref[c, :width - nmom] = pack(scale * (np.abs(blk[:, :d]).T @ np.abs(blk)), d, W)
        if moments:
            ref[c, width - nmom:] = blk.sum(axis=0)
            absref[c, width - nmom:] = np.abs(blk).sum(axis=0)
    return ref, absref


def normalized_error(partials, ref, abs_ref):
    """max over entries of |partial - ref| / sum |a| |b|.  An entry whose absolute sum is 0 (a sigma = 0
    regressor, an empty chunk, the moments of a non-centred launch) must be exactly 0; NaN counts as inf."""
    p = np.asarray(partials, dtype=np.float64)
    err = np.abs(p - ref)
    out = np.where(abs_ref > 0, err / np.where(abs_ref > 0, abs_ref, 1.0), np.where(err == 0, 0.0, np.inf))
    out = np.where(np.isfinite(p), out, np.inf)
    return float(out.max()) if out.size else 0.0


# --------------------------------------------------------------------------------------------------
# error models of the two Gram engines
# --------------------------------------------------------------------------------------------------
def bf16(x):
    """float32 -> bf16 (round to nearest even), returned as float32."""
    b = np.asarray(x, dtype=F32).view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) & 0xFFFF0000).astype(np.uint32).view(F32)


def _model_chunks(rows, N, C, S, d, paired, block_fn):
    r = np.asarray(rows, dtype=F32)
    W = r.shape[1]
    out = []
    for lo, hi in chunk_bounds(N, C, S, paired):
        G = block_fn(r[lo:hi], d).astype(np.float64)
        if paired:
            G[:, :d] *= 2.0
        out.append(pack(G, d, W))
    return np.array(out)


def _ffma_block(blk, d, threads=128):
    """CUDA-core engine: thread t sums the samples t, t + 128, ... in float32, then a pairwise float32 tree."""
    K = (blk.shape[0] + threads - 1) // threads
    pad = np.zeros((K * threads, blk.shape[1]), dtype=F32)
    pad[:blk.shape[0]] = blk
    pad = pad.reshape(K, threads, -1)
    acc = np.zeros((threads, d, blk.shape[1]), dtype=F32)
    for k in range(K):
        acc = (acc + (pad[k][:, :d, None] * pad[k][:, None, :]).astype(F32)).astype(F32)
    while acc.shape[0] > 1:
        acc = (acc[0::2] + acc[1::2]).astype(F32)
    return acc[0]


def _tc_block(blk, d, k=16):
    """Tensor-core engine: every value split into bf16 pieces hi + lo, the piece products exact, float32
    accumulation per K = 16 block of samples."""
    hi = bf16(blk)
    lo = bf16((blk - hi).astype(F32))
    v = hi.astype(np.float64) + lo.astype(np.float64)
    acc = np.zeros((d, blk.shape[1]), dtype=F32)
    for s in range(0, blk.shape[0], k):
        r = v[s:s + k]
        acc = (acc + (r[:, :d].T @ r).astype(F32)).astype(F32)
    return acc


def ffma_model(rows, N, C, S, d, paired=False):
    return _model_chunks(rows, N, C, S, d, paired, _ffma_block)


def tc_model(rows, N, C, S, d, paired=False):
    return _model_chunks(rows, N, C, S, d, paired, _tc_block)


# --------------------------------------------------------------------------------------------------
# kernel-bug mutations: each returns the float64 partials a kernel with that bug would write
# --------------------------------------------------------------------------------------------------
def _bounds_with(N, C, S, paired, fn):
    return [fn(c, lo, hi) for c, (lo, hi) in enumerate(chunk_bounds(N, C, S, paired))]


def mutate_drop_sample(rows, N, C, S, d, paired=False, moments=None):
    """The last row of every chunk is skipped (an off-by-one end: s_end - 1)."""
    b = _bounds_with(N, C, S, paired, lambda c, lo, hi: (lo, max(lo, hi - 1)))
    return chunk_partials(rows, N, C, S, d, paired, moments, bounds=b)[0]


def mutate_duplicate_sample(rows, N, C, S, d, paired=False, moments=None):
    """The first row of every chunk is counted twice."""
    r = np.asarray(rows)
    ref = chunk_partials(r, N, C, S, d, paired, moments)[0]
    first = [lo for lo, _ in chunk_bounds(N, C, S, paired)]
    extra = chunk_partials(r[first], N, C, S, d, paired, moments, bounds=[(k, k + 1) for k in range(C)])[0]
    return ref + extra


def mutate_shift_boundary(rows, N, C, S, d, paired=False, moments=None):
    """Chunk c starts one row late and ends one row late (the chunk boundary moved by one)."""
    R = np.asarray(rows).shape[0]
    b = _bounds_with(N, C, S, paired, lambda c, lo, hi: (min(lo + 1, R), min(hi + 1, R)))
    return chunk_partials(rows, N, C, S, d, paired, moments, bounds=b)[0]


def mutate_hi_only(rows, N, C, S, d, paired=False, moments=None):
    """Tensor-core split without the lo piece: every value rounded to bf16."""
    return chunk_partials(bf16(rows), N, C, S, d, paired, moments)[0]


def mutate_regressor_for_response(rows, N, C, S, d, paired=False, moments=None):
    """Response column 0 staged from regressor column 0 (an operand-row index mix-up)."""
    r = np.array(rows)
    r[:, d] = r[:, 0]
    return chunk_partials(r, N, C, S, d, paired, moments)[0]


def mutate_moment_off_by_one(rows, N, C, S, d, paired=False, moments=None):
    """The first moments of every chunk miss its last row (the Gram itself is right)."""
    ref = chunk_partials(rows, N, C, S, d, paired, moments)[0]
    b = _bounds_with(N, C, S, paired, lambda c, lo, hi: (lo, max(lo, hi - 1)))
    short = chunk_partials(rows, N, C, S, d, paired, moments, bounds=b)[0]
    nmom = np.asarray(rows).shape[1]      # d + n slots: [z' | dF]
    ref[:, -nmom:] = short[:, -nmom:]
    return ref


def mutate_lone_unscaled(w, f, fbar, N, C, S, d):
    """Paired rows whose lone + member keeps its response unscaled: [z / sqrt 2 | f+ - fbar]."""
    r = paired_rows(w, f, fbar)
    if N % 2:
        r[-1, d:] = (np.asarray(f, dtype=F32)[-1] - np.asarray(fbar, dtype=F32)).astype(F32)
    return chunk_partials(r, N, C, S, d, paired=True)[0]


def mutate_pair_sign(w, f, fbar, N, C, S, d):
    """Paired rows staged as [z | f- - f+]."""
    r = paired_rows(w, f, fbar)
    q = N // 2
    r[:q, d:] = -r[:q, d:]
    return chunk_partials(r, N, C, S, d, paired=True)[0]


ROW_MUTATIONS = {
    "drop a sample": mutate_drop_sample,
    "duplicate a sample": mutate_duplicate_sample,
    "chunk boundary moved by one": mutate_shift_boundary,
    "hi piece only": mutate_hi_only,
    "regressor row in place of a response row": mutate_regressor_for_response,
}
PAIR_MUTATIONS = {
    "lone member unscaled": mutate_lone_unscaled,
    "pair sign swapped": mutate_pair_sign,
}
