// TVLQR for state and input dimensions given at run time (1 <= n, m <= kTvlqrAnyMaxDim): solve_tvlqr on a
// linearization of any system, not only of the built-in ones.  The kernels of tvlqr.cuh and tvlqr_box.cuh are
// unrolled over compile-time (n, m) and instantiated for the built-in pairs; the three kernels here take n and
// m as arguments and size their shared memory from them.  Same problem, same conventions:
//
//   tvlqr_riccati_any_kernel   the backward recursion of tvlqr_riccati_kernel (R halved, sym(Q), sym(Qd),
//                              sym(R); H symmetrised before it is factored; P_t written as the mean of (i,j)
//                              and (j,i)), one block per instance.  H is factored by an fp64 root-free
//                              Cholesky L D L' (one warp, lane = row, left-looking) and K, k (and H^-1 when
//                              asked for) come from two triangular solves, one right-hand side per thread.
//   linear_rollout_any_kernel  x_{t+1} = A x + B u + c, u = K x + k: one warp per instance, lane = coordinate.
//   box_qp_any_kernel          one box-constrained QP from x0: the ADMM of box_mpc_kernel with mpc = 0.
#pragma once
#include <cuda_pipeline.h>
#include "tvlqr.cuh"

namespace irs {

constexpr int kTvlqrAnyMaxDim = 32;          // one lane per coordinate in the warp-wide vector sweeps
constexpr int kTvlqrAnyMaxThreads = 256;

// Threads of the Riccati block: one warp per 32 outputs of the widest phase (PA, PB, w), 1 to 8 warps.  Small
// problems keep their barriers cheap; the block size does not change any result.
inline int tvlqr_any_threads(int n, int m) {
    const int warps = (n * n + n * m + n + 31) / 32;
    return 32 * (warps < 1 ? 1 : (warps > kTvlqrAnyMaxThreads / 32 ? kTvlqrAnyMaxThreads / 32 : warps));
}

// Shared-memory layout of tvlqr_riccati_any_kernel, in doubles.  X holds the solutions of H X = -[G | g] and,
// when H^-1 is asked for, H X = I: m rows of n + 1 + m columns.  H is factored in place (L D L': L in its lower
// triangle, L D in its upper one, D on the diagonal).  A, B, c, xd have two slots: step t - 1's operands are
// copied in while step t is computed.
struct TvlqrAnyLayout {
    int nn, nm, mm, ncol;
    int P, Qs, PA, A, B, PB, G, X, H, rd, w, c, xd, g, total;      // slot s of P, A, B, c, xd: + s * its size
    __host__ __device__ TvlqrAnyLayout(int n, int m) {
        nn = n * n;  nm = n * m;  mm = m * m;  ncol = n + 1 + m;
        int o = 0;
        P = o;  o += 2 * (nn + n);     // P then p, ping-pong between steps
        Qs = o;  o += nn;
        PA = o;  o += nn;
        A = o;  o += 2 * nn;
        B = o;  o += 2 * nm;
        PB = o;  o += nm;
        G = o;  o += nm;
        X = o;  o += m * ncol;
        H = o;  o += mm;
        rd = o;  o += m;
        w = o;  o += n;
        c = o;  o += 2 * n;
        xd = o;  o += 2 * n;
        g = o;  o += m;
        total = o;
    }
};

inline size_t tvlqr_riccati_any_smem_bytes(int n, int m) { return sizeof(double) * (size_t)TvlqrAnyLayout(n, m).total; }

// sum_{q<len} a[q*sa] * b[q*sb] + init with four partial sums, term q into sum q % 4: the summation order of dot4
__device__ __forceinline__ double dot_any(const double* a, int sa, const double* b, int sb, int len, double init = 0.0) {
    double acc0 = init, acc1 = 0.0, acc2 = 0.0, acc3 = 0.0;
    int q = 0;
    for (; q + 4 <= len; q += 4) {
        acc0 += a[q * sa] * b[q * sb];
        acc1 += a[(q + 1) * sa] * b[(q + 1) * sb];
        acc2 += a[(q + 2) * sa] * b[(q + 2) * sb];
        acc3 += a[(q + 3) * sa] * b[(q + 3) * sb];
    }
    if (q < len) acc0 += a[q * sa] * b[q * sb];
    if (q + 1 < len) acc1 += a[(q + 1) * sa] * b[(q + 1) * sb];
    if (q + 2 < len) acc2 += a[(q + 2) * sa] * b[(q + 2) * sb];
    return (acc0 + acc1) + (acc2 + acc3);
}

struct TvlqrAnyArgs {
    TvlqrArgs a;     // K, k, status, Hinv, Pout as in tvlqr_riccati_kernel; t_lo, t_hi, carry unused
    int n, m;
};

__global__ void __launch_bounds__(kTvlqrAnyMaxThreads) tvlqr_riccati_any_kernel(const TvlqrAnyArgs args) {
    extern __shared__ __align__(16) double sm_any[];
    const TvlqrArgs& a = args.a;
    const int n = args.n, m = args.m;
    const TvlqrAnyLayout L(n, m);
    const int nn = L.nn, nm = L.nm, mm = L.mm;
    const int G = blockDim.x, gt = threadIdx.x, lane = gt & 31;
    const int inst = blockIdx.x;
    const bool want_hinv = a.Hinv != nullptr;
    const int ncol = want_hinv ? n + 1 + m : n + 1;     // right-hand sides of the solves
    const int ld = L.ncol;                              // row stride of X
    double* Qs = sm_any + L.Qs;
    double* PA = sm_any + L.PA;
    double* PB = sm_any + L.PB;
    double* Gm = sm_any + L.G;
    double* X = sm_any + L.X;
    double* H = sm_any + L.H;
    double* rd = sm_any + L.rd;
    double* w = sm_any + L.w;
    double* g = sm_any + L.g;
    const double* xd_i = a.xd + inst * a.xd_stride;
    bool ok = true;
    // step t's A, B, c, xd into slot s, asynchronously (cp.async): the copy overlaps the step being computed
    auto prefetch = [&](int t, int s) {
        const long long it = (long long)inst * a.T + t;
        for (int e = gt; e < nn; e += G) __pipeline_memcpy_async(sm_any + L.A + s * nn + e, a.At + it * nn + e, sizeof(double));
        for (int e = gt; e < nm; e += G) __pipeline_memcpy_async(sm_any + L.B + s * nm + e, a.Bt + it * nm + e, sizeof(double));
        for (int e = gt; e < n; e += G) {
            __pipeline_memcpy_async(sm_any + L.c + s * n + e, a.ct + it * n + e, sizeof(double));
            __pipeline_memcpy_async(sm_any + L.xd + s * n + e, xd_i + (long long)t * n + e, sizeof(double));
        }
        __pipeline_commit();
    };
    prefetch(a.T - 1, 0);
    // terminal condition: P_T = sym(Qd), p_T = -sym(Qd) xd_T; sym(Q) for the recursion
    {
        double* P = sm_any + L.P;
        for (int e = gt; e < nn; e += G) {
            const int i = e / n, j = e % n;
            const double qd = 0.5 * (a.Qd[e] + a.Qd[j * n + i]);
            P[e] = qd;
            Qs[e] = 0.5 * (a.Q[e] + a.Q[j * n + i]);
            if (a.Pout != nullptr) a.Pout[((long long)inst * (a.T + 1) + a.T) * nn + e] = qd;
        }
        for (int i = gt; i < n; i += G) {
            double acc = 0.0;
            for (int q = 0; q < n; ++q) acc -= 0.5 * (a.Qd[i * n + q] + a.Qd[q * n + i]) * xd_i[(long long)a.T * n + q];
            P[nn + i] = acc;
        }
    }
    int cur = 0;      // operand slot and P buffer of the current step
    for (int t = a.T - 1; t >= 0; --t) {
        const long long it = (long long)inst * a.T + t;
        __pipeline_wait_prior(0);
        __syncthreads();
        if (t > 0) prefetch(t - 1, cur ^ 1);
        const double* A = sm_any + L.A + cur * nn;
        const double* B = sm_any + L.B + cur * nm;
        const double* c = sm_any + L.c + cur * n;
        const double* xd = sm_any + L.xd + cur * n;
        const double* P = sm_any + L.P + cur * (nn + n);
        const double* p = P + nn;
        double* Pn = sm_any + L.P + (cur ^ 1) * (nn + n);
        // PA = P A, PB = P B, w = P c + p
        for (int e = gt; e < nn + nm + n; e += G) {
            if (e < nn) {
                const int i = e / n, j = e % n;
                PA[e] = dot_any(&P[i * n], 1, &A[j], n, n);
            } else if (e < nn + nm) {
                const int f = e - nn, i = f / m, j = f % m;
                PB[f] = dot_any(&P[i * n], 1, &B[j], m, n);
            } else {
                const int i = e - nn - nm;
                w[i] = dot_any(&P[i * n], 1, c, 1, n, p[i]);
            }
        }
        __syncthreads();
        // H = R/2 + B'PB, G = B'PA, g = B'w
        for (int e = gt; e < mm + nm + m; e += G) {
            if (e < mm) {
                const int i = e / m, j = e % m;
                H[e] = dot_any(&B[i], m, &PB[j], m, n, 0.5 * a.R[e]);
            } else if (e < mm + nm) {
                const int f = e - mm, i = f / n, j = f % n;
                Gm[f] = dot_any(&B[i], m, &PA[j], n, n);
            } else {
                const int i = e - mm - nm;
                g[i] = dot_any(&B[i], m, w, 1, n);
            }
        }
        __syncthreads();
        // root-free Cholesky sym(H) = L D L' (L unit lower) by the first warp, left-looking, lane r = row r.  L_rj
        // overwrites H's lower triangle, the unscaled column C_rj = L_rj d_j its upper triangle at (j, r) (each entry
        // of sym(H) is read before lane r replaces it), d_j its diagonal; rd = 1 / d by the reciprocal of
        // spd_inverse.  Lane r reads its C_rk down a column: consecutive lanes, consecutive words.
        if (gt < 32) {
            for (int j = 0; j < m; ++j) {
                double s = 0.0;
                if (lane >= j && lane < m)
                    s = 0.5 * (H[lane * m + j] + H[j * m + lane]) - dot_any(&H[lane], m, &H[j * m], 1, j);
                const double d = __shfl_sync(0xffffffffu, s, j);
                const bool pivot = d > 0.0;                  // false for NaN too
                ok = ok && pivot;
                const double r = fast_rcp(pivot ? d : 1.0);
                if (lane == j) {
                    H[j * m + j] = d;
                    rd[j] = r;
                } else if (lane > j && lane < m) {
                    H[j * m + lane] = s;
                    H[lane * m + j] = s * r;
                }
                __syncwarp();
            }
        }
        __syncthreads();
        // one right-hand side per thread, in place in column `col` of X: L y = b, then L' x = D^-1 y.
        // b = -G[:, col] (K_t), -g (k_t) or e_j (column j of H^-1).  For m = 1 this is b / H exactly as the templated
        // kernel forms it (fast_rcp(H) b).
        for (int col = gt; col < ncol; col += G) {
            for (int i = 0; i < m; ++i) {
                const double b = col < n ? -Gm[i * n + col] : (col == n ? -g[i] : (col - n - 1 == i ? 1.0 : 0.0));
                X[i * ld + col] = b - dot_any(&H[i * m], 1, &X[col], ld, i);
            }
            for (int i = m - 1; i >= 0; --i)
                X[i * ld + col] = X[i * ld + col] * rd[i] - dot_any(&H[(i + 1) * m + i], m, &X[(i + 1) * ld + col], ld, m - 1 - i);
            if (col < n) {
                for (int i = 0; i < m; ++i) {
                    const double y = X[i * ld + col];
                    a.K[(it * m + i) * n + col] = y;
                    ok = ok && isfinite(y);
                }
            } else if (col == n) {
                for (int i = 0; i < m; ++i) {
                    const double y = X[i * ld + n];
                    a.k[it * m + i] = y;
                    ok = ok && isfinite(y);      // NaN / Inf in c or xd reach k only
                }
            }
        }
        __syncthreads();
        if (want_hinv)
            for (int e = gt; e < mm; e += G) {
                const int i = e / m, j = e % m;
                a.Hinv[it * mm + e] = 0.5 * (X[i * ld + n + 1 + j] + X[j * ld + n + 1 + i]);
            }
        // P <- sym(Q + A'PA + G'K),  p <- -sym(Q) xd_t + A'w + G'k, into the other buffer (entry (i,j) and its mirror
        // formed as in tvlqr_riccati_kernel, Q as given: the mean of the two is sym(Q) + sym(A'PA + G'K))
        for (int e = gt; e < nn + n; e += G) {
            if (e < nn) {
                const int i = e / n, j = e % n;
                const double aij = dot_any(&A[i], n, &PA[j], n, n, a.Q[i * n + j]) + dot_any(&Gm[i], n, &X[j], ld, m);
                const double aji = dot_any(&A[j], n, &PA[i], n, n, a.Q[j * n + i]) + dot_any(&Gm[j], n, &X[i], ld, m);
                const double v = 0.5 * (aij + aji);
                Pn[e] = v;
                if (a.Pout != nullptr) a.Pout[((long long)inst * (a.T + 1) + t) * nn + e] = v;
            } else {
                const int i = e - nn;
                Pn[e] = (dot_any(&A[i], n, w, 1, n) - dot_any(&Qs[i * n], 1, xd, 1, n)) + dot_any(&Gm[i], n, &X[n], ld, m);
            }
        }
        cur ^= 1;
        // (the barrier at the top of the next step orders these writes before their reads)
    }
    __syncthreads();
    // NaN guard on the final value function (every K_t, k_t has been checked where it was written)
    const double* P = sm_any + L.P + cur * (nn + n);
    for (int e = gt; e < nn; e += G)
        if (!(P[e] == P[e])) ok = false;
    ok = __syncthreads_and(ok);
    if (gt == 0) a.status[inst] = ok ? 0 : 1;
}

// x_{t+1} = A_t x_t + B_t u_t + c_t, u_t = K_t x_t + k_t from x0 [I, n]: one warp per instance, lanes = coordinates
constexpr int kRolloutAnyWarps = 4;

__global__ void __launch_bounds__(32 * kRolloutAnyWarps) linear_rollout_any_kernel(const TvlqrArgs a, int n, int m,
                                                                                   const double* x0, double* xs,
                                                                                   double* us) {
    __shared__ double xv[kRolloutAnyWarps][kTvlqrAnyMaxDim], uv[kRolloutAnyWarps][kTvlqrAnyMaxDim];
    const int sub = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inst = blockIdx.x * kRolloutAnyWarps + sub;
    if (inst >= a.I) return;      // whole warp exits together
    double* x = xv[sub];
    double* u = uv[sub];
    if (lane < n) {
        x[lane] = x0[(long long)inst * n + lane];
        xs[(long long)inst * (a.T + 1) * n + lane] = x[lane];
    }
    __syncwarp();
    for (int t = 0; t < a.T; ++t) {
        const long long it = (long long)inst * a.T + t;
        if (lane < m) {
            const double v = dot_any(a.K + (it * m + lane) * n, 1, x, 1, n, a.k[it * m + lane]);
            u[lane] = v;
            us[it * m + lane] = v;
        }
        __syncwarp();
        double xn = 0.0;
        if (lane < n)
            xn = dot_any(a.Bt + (it * n + lane) * m, 1, u, 1, m, dot_any(a.At + (it * n + lane) * n, 1, x, 1, n, a.ct[it * n + lane]));
        __syncwarp();
        if (lane < n) {
            x[lane] = xn;
            xs[((long long)inst * (a.T + 1) + t + 1) * n + lane] = xn;
        }
        __syncwarp();
    }
}

struct BoxQpAnyArgs {
    const double* At;     // [I, T, n, n]
    const double* Bt;     // [I, T, n, m]
    const double* ct;     // [I, T, n]
    const double* K;      // [I, T, m, n]   gains of the penalty-augmented problem
    const double* Hinv;   // [I, T, m, m]
    const double* P;      // [I, T+1, n, n]
    const double* Q;      // [n, n]  (original weights)
    const double* Qd;
    const double* xd;     // [I or 1, T+1, n]
    long long xd_stride;
    const double* dx;     // [n] ADMM penalties on the states
    const double* du;     // [m] ... on the inputs
    const double* xlo;    // [n], or [T+1, n] when xbox_stride = n
    const double* xhi;
    const double* ulo;    // [m], or [T, m] when ubox_stride = m
    const double* uhi;
    long long xbox_stride, ubox_stride;
    const double* x0;     // [I, n]
    double alpha, eps;
    int max_iter;
    double* x_trj;        // [I, T+1, n]
    double* u_trj;        // [I, T, m]
    int* status;          // [I] 0 ok, 1 ADMM did not converge / NaN
    int* iters;           // [I] ADMM iterations
    int I, T, n, m;
};

// Dynamic shared memory of box_qp_any_kernel in doubles: the layout of box_mpc_smem_bytes, and with CACHE the
// per-step A_t, B_t, K_t, Hinv_t, c_t (box_mpc_kernel's cache less the skip path's K0_t, k0_t, which one QP
// from x0 never reads).
inline size_t box_qp_any_smem_bytes(int n, int m, int T, bool cache) {
    size_t d = (size_t)3 * (T + 1) * n + (size_t)4 * T * m + (size_t)T * n + (size_t)(T + 1) * n + 2 * n + n + m;
    if (cache) d += (size_t)T * (n * n + 2 * n * m + m * m + n);
    return sizeof(double) * d;
}

// One warp per instance; lanes = coordinates.  The algorithm, its cold start and its stopping rule are those of
// box_mpc_kernel with mpc = 0 (see there and oracle/box_tvlqr.py), with loops over the run-time n and m.
template <bool CACHE>
__global__ void __launch_bounds__(32) box_qp_any_kernel(const BoxQpAnyArgs a) {
    extern __shared__ __align__(16) double sm_box[];
    const int T = a.T, n = a.n, m = a.m;
    double* zx = sm_box;
    double* wx = zx + (T + 1) * n;
    double* x = wx + (T + 1) * n;
    double* zu = x + (T + 1) * n;
    double* wu = zu + T * m;
    double* u = wu + T * m;
    double* kk = u + T * m;
    double* Pc = kk + T * m;
    double* qxd = Pc + T * n;         // sym(Q) xd_t (t < T), sym(Qd) xd_T
    double* pv = qxd + (T + 1) * n;   // [2][n] rolling p_{t+1}, p_t
    double* ww = pv + 2 * n;          // [n]
    double* gv = ww + n;              // [m]
    double* cache = gv + m;
    const int lane = threadIdx.x;
    const int inst = blockIdx.x;
    const long long base = (long long)inst * T;
    const double* xd_i = a.xd + inst * a.xd_stride;
    const double dxl = lane < n ? a.dx[lane] : 0.0, dul = lane < m ? a.du[lane] : 0.0;
    const double* Ap = a.At + base * n * n;
    const double* Bp = a.Bt + base * n * m;
    const double* Kp = a.K + base * m * n;
    const double* Hp = a.Hinv + base * m * m;
    const double* cp = a.ct + base * n;
    if constexpr (CACHE) {
        double* sA = cache;
        double* sB = sA + T * n * n;
        double* sK = sB + T * n * m;
        double* sH = sK + T * m * n;
        double* sc = sH + T * m * m;
        for (int e = lane; e < T * n * n; e += 32) sA[e] = Ap[e];
        for (int e = lane; e < T * n * m; e += 32) { sB[e] = Bp[e];  sK[e] = Kp[e]; }
        for (int e = lane; e < T * m * m; e += 32) sH[e] = Hp[e];
        for (int e = lane; e < T * n; e += 32) sc[e] = cp[e];
        Ap = sA;  Bp = sB;  Kp = sK;  Hp = sH;  cp = sc;
    }
    // Pc_t = P_{t+1} c_t, sym(Q) xd_t, sym(Qd) xd_T; cold start of the split variables: z = clip(target), w = 0
    for (int e = lane; e < T * n; e += 32) {
        const int t = e / n, i = e % n;
        const double* Pr = a.P + ((long long)inst * (T + 1) + t + 1) * n * n + i * n;
        double acc = 0.0, accq = 0.0;
        for (int q = 0; q < n; ++q) {
            acc += Pr[q] * a.ct[(base + t) * n + q];
            accq += 0.5 * (a.Q[i * n + q] + a.Q[q * n + i]) * xd_i[(long long)t * n + q];
        }
        Pc[e] = acc;
        qxd[e] = accq;
    }
    if (lane < n) {
        double accq = 0.0;
        for (int q = 0; q < n; ++q) accq += 0.5 * (a.Qd[lane * n + q] + a.Qd[q * n + lane]) * xd_i[(long long)T * n + q];
        qxd[T * n + lane] = accq;
    }
    for (int e = lane; e < (T + 1) * n; e += 32) {
        const int i = e % n;
        zx[e] = fmin(fmax(xd_i[e], a.xlo[(e / n) * a.xbox_stride + i]), a.xhi[(e / n) * a.xbox_stride + i]);
        wx[e] = 0.0;
        x[e] = 0.0;
    }
    for (int e = lane; e < T * m; e += 32) {
        const int j = e % m;
        zu[e] = fmin(fmax(0.0, a.ulo[(e / m) * a.ubox_stride + j]), a.uhi[(e / m) * a.ubox_stride + j]);
        wu[e] = 0.0;
        u[e] = 0.0;
    }
    if (lane < n) x[lane] = a.x0[(long long)inst * n + lane];
    __syncwarp();
    int iters = 0;
    bool converged = false;
    for (int it = 0; it < a.max_iter && !converged; ++it) {
        // ---- backward vector recursion: p_T, then kk_t, p_t for t = T-1 .. 0 ----
        int cur = 0;
        if (lane < n) pv[lane] = -(qxd[T * n + lane] + 0.5 * dxl * (zx[T * n + lane] - wx[T * n + lane]));
        __syncwarp();
        for (int t = T - 1; t >= 0; --t) {
            if (lane < n) ww[lane] = Pc[t * n + lane] + pv[cur * n + lane];
            __syncwarp();
            if (lane < m) {
                double g = -0.5 * dul * (zu[t * m + lane] - wu[t * m + lane]);
                const double* Bc = Bp + t * n * m + lane;
                for (int q = 0; q < n; ++q) g += Bc[q * m] * ww[q];
                gv[lane] = g;
            }
            __syncwarp();
            if (lane < m) {
                const double* Hr = Hp + (t * m + lane) * m;
                double acc = 0.0;
                for (int q = 0; q < m; ++q) acc -= Hr[q] * gv[q];
                kk[t * m + lane] = acc;
            }
            if (t > 0 && lane < n) {
                double acc = -(qxd[t * n + lane] + 0.5 * dxl * (zx[t * n + lane] - wx[t * n + lane]));
                const double* Ac = Ap + t * n * n + lane;
                for (int q = 0; q < n; ++q) acc += Ac[q * n] * ww[q];
                const double* Kc = Kp + t * m * n + lane;
                for (int q = 0; q < m; ++q) acc += Kc[q * n] * gv[q];
                pv[(cur ^ 1) * n + lane] = acc;
            }
            cur ^= 1;
            __syncwarp();
        }
        // ---- forward affine rollout from the fixed x_0 ----
        for (int t = 0; t < T; ++t) {
            if (lane < m) {
                const double* Kr = Kp + (t * m + lane) * n;
                double acc = kk[t * m + lane];
                for (int q = 0; q < n; ++q) acc += Kr[q] * x[t * n + q];
                u[t * m + lane] = acc;
            }
            __syncwarp();
            if (lane < n) {
                const double* Ar = Ap + (t * n + lane) * n;
                const double* Br = Bp + (t * n + lane) * m;
                double acc = cp[t * n + lane];
                for (int q = 0; q < n; ++q) acc += Ar[q] * x[t * n + q];
                for (int q = 0; q < m; ++q) acc += Br[q] * u[t * m + q];
                x[(t + 1) * n + lane] = acc;
            }
            __syncwarp();
        }
        // ---- relaxed projection, dual update, residuals in the units of z ----
        double r_prim = 0.0, r_dual = 0.0, scale = 1.0;
        for (int e = n + lane; e < (T + 1) * n; e += 32) {
            const int i = e % n;
            const double xh = a.alpha * x[e] + (1.0 - a.alpha) * zx[e];
            const double zn = fmin(fmax(xh + wx[e], a.xlo[(e / n) * a.xbox_stride + i]), a.xhi[(e / n) * a.xbox_stride + i]);
            wx[e] += xh - zn;
            r_prim = fmax(r_prim, fabs(x[e] - zn));
            r_dual = fmax(r_dual, fabs(zn - zx[e]));
            scale = fmax(scale, fabs(zn));
            zx[e] = zn;
        }
        for (int e = lane; e < T * m; e += 32) {
            const int j = e % m;
            const double uh = a.alpha * u[e] + (1.0 - a.alpha) * zu[e];
            const double zn = fmin(fmax(uh + wu[e], a.ulo[(e / m) * a.ubox_stride + j]), a.uhi[(e / m) * a.ubox_stride + j]);
            wu[e] += uh - zn;
            r_prim = fmax(r_prim, fabs(u[e] - zn));
            r_dual = fmax(r_dual, fabs(zn - zu[e]));
            scale = fmax(scale, fabs(zn));
            zu[e] = zn;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            r_prim = fmax(r_prim, __shfl_xor_sync(0xffffffffu, r_prim, o));
            r_dual = fmax(r_dual, __shfl_xor_sync(0xffffffffu, r_dual, o));
            scale = fmax(scale, __shfl_xor_sync(0xffffffffu, scale, o));
        }
        ++iters;
        // NaN-safe: a NaN residual never satisfies the test and the solve ends as "failed"
        converged = (r_prim <= a.eps * scale) && (r_dual <= a.eps * scale);
        __syncwarp();
    }
    // the QP plan (states consistent with the dynamics)
    for (int e = lane; e < (T + 1) * n; e += 32) a.x_trj[(long long)inst * (T + 1) * n + e] = x[e];
    for (int e = lane; e < T * m; e += 32) a.u_trj[base * m + e] = u[e];
    if (lane == 0) {
        a.status[inst] = converged ? 0 : 1;
        a.iters[inst] = iters;
    }
}

}  // namespace irs
