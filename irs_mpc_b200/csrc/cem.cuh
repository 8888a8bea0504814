// Cross-entropy-method step on the device (irs_lqr/cem.py:151-184): elite selection and the mean / std
// refit of the candidate input trajectories.  The candidates are rolled out and costed by the batched
// open-loop rollout kernel (tvlqr.cuh); these two kernels replace the reference's np.argpartition and
// np.mean / np.std over the elites, so the B x T x m candidates never travel back to the host.
#pragma once
#include "common.cuh"

namespace irs {

// elite[b] = 1 iff b is among the first n_elite candidates in the order of the key (isnan(cost), cost,
// index): every NaN after every other value, +inf included (as np.argpartition / np.argsort place it, so a
// diverged rollout never displaces an infinite-cost one), equal costs (-0.0 == +0.0) and NaNs by index.
// The rank of b is the number of candidates that come before it in that total order, so exactly n_elite
// are marked.  O(B^2) comparisons, B ~ 1e3-1e4 (the reference uses an O(B) partial partition; any choice
// among equal costs is valid).
__global__ void __launch_bounds__(256) cem_rank_kernel(const double* cost, int B, int n_elite, int* elite) {
    __shared__ double tile[256];
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    const double mine = b < B ? cost[b] : 0.0;
    const bool mine_nan = mine != mine;
    int rank = 0;
    for (int base = 0; base < B; base += 256) {
        const int j = base + threadIdx.x;
        __syncthreads();
        tile[threadIdx.x] = j < B ? cost[j] : 0.0;
        __syncthreads();
        const int lim = B - base < 256 ? B - base : 256;
        for (int q = 0; q < lim; ++q) {
            const double v2 = tile[q];
            const bool nan2 = v2 != v2;
            const bool before = nan2 != mine_nan ? mine_nan                        // the non-NaN one first
                              : nan2 ? base + q < b                                // both NaN: by index
                              : v2 < mine || (v2 == mine && base + q < b);         // by value, then by index
            rank += before ? 1 : 0;
        }
    }
    if (b < B) elite[b] = rank < n_elite ? 1 : 0;
}

// mean[e] and std[e] (population standard deviation, np.std default) of u[b][e] over the elites, one thread
// per coordinate e of the T x m trajectory, elites visited in index order (deterministic).
__global__ void __launch_bounds__(128) cem_refit_kernel(const double* u, const int* elite, int B, int width,
                                                        int n_elite, double* mean, double* std_out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= width) return;
    double s = 0.0;
    for (int b = 0; b < B; ++b)
        if (elite[b]) s += u[(long long)b * width + e];
    const double mu = s / (double)n_elite;
    double v = 0.0;
    for (int b = 0; b < B; ++b)
        if (elite[b]) {
            const double dlt = u[(long long)b * width + e] - mu;
            v = fma(dlt, dlt, v);
        }
    mean[e] = mu;
    std_out[e] = sqrt(v / (double)n_elite);
}

// Packed Gram block [Z^T Z (upper rows) | Z^T F] in fp64 from explicit samples Z [N, d], F [N, n]
// (IrsLqrZeroOrder.compute_least_squares, irs_lqr/irs_lqr_zero_order.py:27-36): entry e = (i, j) of the
// layout the finalize kernel reads (row i holds columns j = i .. d + n - 1), one thread per entry.
__global__ void __launch_bounds__(128) gram_block_f64_kernel(const double* Z, const double* F, long long N,
                                                             int n, int d, double* out) {
    const int W = d + n;
    const int nacc = d * (d + 1) / 2 + d * n;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= nacc) return;
    int i = 0;
    while (i + 1 < d && (i + 1) * W - (i + 1) * i / 2 <= e) ++i;
    const int j = i + (e - (i * W - i * (i - 1) / 2));
    double s = 0.0;
    for (long long k = 0; k < N; ++k) {
        const double zi = Z[k * d + i];
        const double wj = j < d ? Z[k * d + j] : F[k * n + (j - d)];
        s = fma(zi, wj, s);
    }
    out[e] = s;
}

}  // namespace irs
