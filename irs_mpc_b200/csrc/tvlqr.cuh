// Time-varying LQR: backward affine Riccati recursion + closed-loop rollout on the true
// dynamics, one warp per independent MPC instance, fp64 (sequential and latency bound; the
// B200 has full-rate-enough FP64 FMA for this and it keeps the cost curves at round-off of the
// reference's float64).
//
// Replaces the T re-solved QPs of irs_lqr/irs_lqr.py:169-184 + irs_lqr/tv_lqr.py:69-137:
//   cost  sum_{s<T} (x_s-xd_s)'Q(x_s-xd_s) + 1/2 u_s'R u_s + (x_T-xd_T)'Qd(x_T-xd_T)
//   s.t.  x_{s+1} = A_s x_s + B_s u_s + c_s
// (Drake's AddQuadraticCost(R,0,u) is 1/2 u'Ru, tv_lqr.py:110).  With inactive bounds the first
// input of every re-solved QP is u_t = K_t x_t + k_t from ONE backward pass (Bellman).
#pragma once
#include "systems.cuh"

namespace irs {

struct TvlqrArgs {
    const double* At;    // [I, T, n, n]
    const double* Bt;    // [I, T, n, m]
    const double* ct;    // [I, T, n]
    const double* Q;     // [n, n]
    const double* Qd;    // [n, n]
    const double* R;     // [m, m]  (full R; halved inside, tv_lqr.py:110)
    const double* xd;    // [I or 1, T+1, n]
    long long xd_stride; // 0 when one desired trajectory is shared by all instances
    double* K;           // [I, T, m, n]
    double* k;           // [I, T, m]
    int* status;         // [I] 0 ok, 1 H not SPD / NaN
    int I, T;
    double* Hinv;        // optional [I, T, m, m]: (R/2 + B'PB)^-1 of every step (bounded solve)
    double* Pout;        // optional [I, T+1, n, n]: value-function Hessians P_t
    // Segment of the recursion (tiled kernel only): steps t_hi-1 .. t_lo.  t_hi == 0 means the whole
    // horizon.  A segment that does not start at T reads (P, p) of step t_hi from carry [I, n*n + n];
    // one that does not end at 0 writes (P, p) of step t_lo there.  Splitting the pass this way lets
    // the late timesteps be solved while the early ones are still being linearized.
    int t_lo, t_hi;
    double* carry;
};

// Reciprocal in fp64 from the hardware seed (MUFU.RCP64H, ~20 bits) and two Newton steps — a
// 5-deep dependent chain instead of the library division's ~12 plus slow-path branches.  The fp64
// special functions sit on the sequential critical path of the recursion.
__device__ __forceinline__ double fast_rcp(double a) {
    double x;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(a));
    x = fma(x, fma(-a, x, 1.0), x);
    x = fma(x, fma(-a, x, 1.0), x);
    return x;
}

// Inverse of a symmetric positive definite m x m matrix (m in {1, 2, 4}) in registers, by 2 x 2
// block elimination: H = [[A, B], [B', D]], S = D - B' A^-1 B.  Two sequential reciprocals for
// m = 4 against four rsqrt + substitutions for a Cholesky solve.  Returns false if H is not SPD
// (Sylvester: A > 0 and S > 0) or contains NaN.
__device__ __forceinline__ bool spd_inverse2(double a, double b, double d, double& ia, double& ib, double& id) {
    const double det = a * d - b * b;
    const bool ok = (a > 0.0) && (det > 0.0);
    const double r = fast_rcp(ok ? det : 1.0);
    ia = d * r;  ib = -b * r;  id = a * r;
    return ok;
}
template <int m>
__device__ __forceinline__ bool spd_inverse(const double (&H)[m][m], double (&Hi)[m][m]) {
    static_assert(m == 1 || m == 2 || m == 4, "input dimensions of the built-in systems");
    if constexpr (m == 1) {
        const bool ok = H[0][0] > 0.0;
        Hi[0][0] = fast_rcp(ok ? H[0][0] : 1.0);
        return ok;
    } else if constexpr (m == 2) {
        const bool ok = spd_inverse2(H[0][0], H[0][1], H[1][1], Hi[0][0], Hi[0][1], Hi[1][1]);
        Hi[1][0] = Hi[0][1];
        return ok;
    } else {
        double a0, a1, a2;                                  // A^-1 = [[a0, a1], [a1, a2]]
        bool ok = spd_inverse2(H[0][0], H[0][1], H[1][1], a0, a1, a2);
        // X = A^-1 B,  B = H[0:2, 2:4]
        const double x00 = a0 * H[0][2] + a1 * H[1][2], x01 = a0 * H[0][3] + a1 * H[1][3];
        const double x10 = a1 * H[0][2] + a2 * H[1][2], x11 = a1 * H[0][3] + a2 * H[1][3];
        // S = D - B' X (symmetric)
        const double s00 = H[2][2] - (H[0][2] * x00 + H[1][2] * x10);
        const double s01 = H[2][3] - (H[0][2] * x01 + H[1][2] * x11);
        const double s11 = H[3][3] - (H[0][3] * x01 + H[1][3] * x11);
        double t0, t1, t2;                                  // S^-1
        ok = spd_inverse2(s00, s01, s11, t0, t1, t2) && ok;
        // Y = X S^-1
        const double y00 = x00 * t0 + x01 * t1, y01 = x00 * t1 + x01 * t2;
        const double y10 = x10 * t0 + x11 * t1, y11 = x10 * t1 + x11 * t2;
        Hi[2][2] = t0;  Hi[2][3] = t1;  Hi[3][2] = t1;  Hi[3][3] = t2;
        Hi[0][2] = -y00;  Hi[0][3] = -y01;  Hi[1][2] = -y10;  Hi[1][3] = -y11;
        Hi[2][0] = -y00;  Hi[3][0] = -y01;  Hi[2][1] = -y10;  Hi[3][1] = -y11;
        Hi[0][0] = a0 + (y00 * x00 + y01 * x01);
        Hi[0][1] = a1 + (y00 * x10 + y01 * x11);
        Hi[1][0] = Hi[0][1];
        Hi[1][1] = a2 + (y10 * x10 + y11 * x11);
        return ok;
    }
}

// sum_{q<len} a[q*sa] * b[q*sb] with four independent partial sums: the fp64 FMA latency, not its
// throughput, bounds the sequential recursion, so the dependent chain is cut from len to len/4 + 2.
template <int len>
__device__ __forceinline__ double dot4(const double* a, int sa, const double* b, int sb, double init = 0.0) {
    double acc[4] = {init, 0.0, 0.0, 0.0};
#pragma unroll
    for (int q = 0; q < len; ++q) acc[q & 3] += a[q * sa] * b[q * sb];
    return (acc[0] + acc[1]) + (acc[2] + acc[3]);
}

template <int n, int m>
struct TvlqrSmem {
    double P[n * n], A[n * n], PA[n * n], Qs[n * n];
    double B[n * m], PB[n * m], G[m * n], Kt[m * n];
    double H[m * m];
    double p[n], w[n], c[n], xd[n], g[m], kt[m];
};

constexpr int kTvlqrWarps = 4;          // warp-per-instance variant: instances per block
constexpr int kTvlqrBlockThreads = 256; // block-per-instance variant

// One cooperative group of G threads per MPC instance: G = 32 (a warp; many instances, throughput)
// or G = blockDim.x (a whole block; few instances, latency).  The step-(t-1) matrices are
// prefetched into registers while step t is computed, so the sequential recursion never waits on
// an exposed global-memory round trip.
template <int n, int m, int G>
__global__ void __launch_bounds__(G == 32 ? 32 * kTvlqrWarps : G) tvlqr_riccati_kernel(const TvlqrArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int sub = G == 32 ? (int)(threadIdx.x >> 5) : 0;      // instance slot inside the block
    const int gt = G == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x;
    const int inst = G == 32 ? blockIdx.x * kTvlqrWarps + sub : blockIdx.x;
    if (inst >= a.I) return;      // whole group exits together
    TvlqrSmem<n, m>& s = reinterpret_cast<TvlqrSmem<n, m>*>(smem_raw)[sub];
    auto group_sync = [] {
        if constexpr (G == 32) __syncwarp();
        else __syncthreads();
    };
    const double* xd_i = a.xd + inst * a.xd_stride;
    bool ok = true;
    // register prefetch slots of this thread
    constexpr int kRA = (n * n + G - 1) / G, kRB = (n * m + G - 1) / G, kRC = (n + G - 1) / G;
    double rA[kRA], rB[kRB], rc[kRC], rxd[kRC];
    auto prefetch = [&](int t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int k = 0; k < kRA; ++k) { const int e = gt + k * G; if (e < n * n) rA[k] = a.At[it * n * n + e]; }
#pragma unroll
        for (int k = 0; k < kRB; ++k) { const int e = gt + k * G; if (e < n * m) rB[k] = a.Bt[it * n * m + e]; }
#pragma unroll
        for (int k = 0; k < kRC; ++k) {
            const int e = gt + k * G;
            if (e < n) { rc[k] = a.ct[it * n + e];  rxd[k] = xd_i[(long long)t * n + e]; }
        }
    };
    prefetch(a.T - 1);
    // terminal condition: P_T = sym(Qd), p_T = -sym(Qd) xd_T; sym(Q) for the gradient term.  The cost
    // x'Qx only sees the symmetric part of a weight, so that is what the recursion uses (for symmetric
    // input 0.5 (a + a) = a exactly: nothing changes).
    for (int e = gt; e < n * n; e += G) {
        const int i = e / n, j = e % n;
        const double qd = 0.5 * (a.Qd[e] + a.Qd[j * n + i]);
        s.P[e] = qd;
        s.Qs[e] = 0.5 * (a.Q[e] + a.Q[j * n + i]);
        if (a.Pout != nullptr) a.Pout[((long long)inst * (a.T + 1) + a.T) * n * n + e] = qd;
    }
    for (int i = gt; i < n; i += G) {
        double acc = 0.0;
        for (int q = 0; q < n; ++q) acc -= 0.5 * (a.Qd[i * n + q] + a.Qd[q * n + i]) * xd_i[(long long)a.T * n + q];
        s.p[i] = acc;
    }
    for (int t = a.T - 1; t >= 0; --t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int k = 0; k < kRA; ++k) { const int e = gt + k * G; if (e < n * n) s.A[e] = rA[k]; }
#pragma unroll
        for (int k = 0; k < kRB; ++k) { const int e = gt + k * G; if (e < n * m) s.B[e] = rB[k]; }
#pragma unroll
        for (int k = 0; k < kRC; ++k) {
            const int e = gt + k * G;
            if (e < n) { s.c[e] = rc[k];  s.xd[e] = rxd[k]; }
        }
        group_sync();
        if (t > 0) prefetch(t - 1);
        // PA = P A, PB = P B, w = P c + p   (one output per thread where G allows)
        for (int e = gt; e < n * n + n * m + n; e += G) {
            if (e < n * n) {
                const int i = e / n, j = e % n;
                s.PA[e] = dot4<n>(&s.P[i * n], 1, &s.A[j], n);
            } else if (e < n * n + n * m) {
                const int f = e - n * n, i = f / m, j = f % m;
                s.PB[f] = dot4<n>(&s.P[i * n], 1, &s.B[j], m);
            } else {
                const int i = e - n * n - n * m;
                s.w[i] = dot4<n>(&s.P[i * n], 1, s.c, 1, s.p[i]);
            }
        }
        group_sync();
        // H = R/2 + B'PB, G = B'PA, g = B'w
        for (int e = gt; e < m * m + m * n + m; e += G) {
            if (e < m * m) {
                const int i = e / m, j = e % m;
                s.H[e] = dot4<n>(&s.B[i], m, &s.PB[j], m, 0.5 * a.R[e]);
            } else if (e < m * m + m * n) {
                const int f = e - m * m, i = f / n, j = f % n;
                s.G[f] = dot4<n>(&s.B[i], m, &s.PA[j], n);
            } else {
                const int i = e - m * m - m * n;
                s.g[i] = dot4<n>(&s.B[i], m, s.w, 1);
            }
        }
        group_sync();
        // the first warp inverts H (m <= 4: registers); threads 0..n-1 form a column of K = -H^-1 G, thread n forms k
        if (gt < 32) {
            double Hs[m][m], Hi[m][m];
#pragma unroll
            for (int i = 0; i < m; ++i)
#pragma unroll
                for (int j = 0; j < m; ++j) Hs[i][j] = 0.5 * (s.H[i * m + j] + s.H[j * m + i]);
            ok = spd_inverse<m>(Hs, Hi) && ok;
            if (a.Hinv != nullptr && gt == 0) {
#pragma unroll
                for (int i = 0; i < m; ++i)
#pragma unroll
                    for (int j = 0; j < m; ++j) a.Hinv[(it * m + i) * m + j] = Hi[i][j];
            }
            for (int col = gt; col <= n; col += G) {
                double b[m], y[m];
#pragma unroll
                for (int i = 0; i < m; ++i) b[i] = col < n ? s.G[i * n + col] : s.g[i];
#pragma unroll
                for (int i = 0; i < m; ++i) {
                    double acc = 0.0;
#pragma unroll
                    for (int q = 0; q < m; ++q) acc -= Hi[i][q] * b[q];
                    y[i] = acc;
                }
                if (col < n) {
#pragma unroll
                    for (int i = 0; i < m; ++i) {
                        s.Kt[i * n + col] = y[i];
                        a.K[(it * m + i) * n + col] = y[i];
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < m; ++i) {
                        s.kt[i] = y[i];
                        a.k[it * m + i] = y[i];
                    }
                }
#pragma unroll
                for (int i = 0; i < m; ++i) ok = ok && isfinite(y[i]);      // NaN / Inf in c or xd reach k only
            }
        }
        group_sync();
        // P <- sym(Q + A'PA + G'K),  p <- -sym(Q) xd_t + A'w + G'k.  Each thread forms entry (i,j) and its
        // mirror (j,i) and writes their mean: P stays exactly symmetric without a second pass.
        double Pnew[(n * n + n + G - 1) / G];
#pragma unroll
        for (int k = 0; k < (n * n + n + G - 1) / G; ++k) {
            const int e = gt + k * G;
            if (e < n * n) {
                const int i = e / n, j = e % n;
                const double aij = dot4<n>(&s.A[i], n, &s.PA[j], n, a.Q[i * n + j]) + dot4<m>(&s.G[i], n, &s.Kt[j], n);
                const double aji = dot4<n>(&s.A[j], n, &s.PA[i], n, a.Q[j * n + i]) + dot4<m>(&s.G[j], n, &s.Kt[i], n);
                Pnew[k] = 0.5 * (aij + aji);
            } else if (e < n * n + n) {
                const int i = e - n * n;
                Pnew[k] = (dot4<n>(&s.A[i], n, s.w, 1) - dot4<n>(&s.Qs[i * n], 1, s.xd, 1)) +
                          dot4<m>(&s.G[i], n, s.kt, 1);
            }
        }
        group_sync();      // everyone has read the old P / p
#pragma unroll
        for (int k = 0; k < (n * n + n + G - 1) / G; ++k) {
            const int e = gt + k * G;
            if (e < n * n) {
                s.P[e] = Pnew[k];
                if (a.Pout != nullptr) a.Pout[((long long)inst * (a.T + 1) + t) * n * n + e] = Pnew[k];
            } else if (e < n * n + n) {
                s.p[e - n * n] = Pnew[k];
            }
        }
        // (the group_sync after the next step's operand stores orders these writes before its reads)
    }
    group_sync();
    // NaN guard on the final value function (every K_t, k_t has been checked where it was written)
    for (int e = gt; e < n * n; e += G)
        if (!(s.P[e] == s.P[e])) ok = false;
    if constexpr (G == 32) {
        ok = __all_sync(0xffffffffu, ok);
    } else {
        ok = __syncthreads_and(ok);
    }
    if (gt == 0) a.status[inst] = ok ? 0 : 1;
}

// ---------------------------------------------------------------------------------------------
// Register-tiled variant for few instances and even n, m (quadrotor 12/4, three_cart 6/2): one block
// of 128 threads per instance, every thread owns a 2 x 2 tile of a matrix product and streams the
// operand rows as 16-byte shared-memory loads (24 LDS.128 for 48 DFMA per tile).  The generic
// kernel above spends most of a step in the LSU: one thread per output needs 2 loads per FMA and
// ~1200 of its ~3150 cycles per step are shared-memory issue; tiling halves the loads per FMA
// twice over (2 x 2 tile, 128-bit loads).
// ---------------------------------------------------------------------------------------------
constexpr int kTvlqrTiledThreads = 128;

template <int n, int m>
struct TvlqrTiledSmem {
    double P[n * n], A[n * n], PA[n * n], Pn[n * n], Q[n * n];
    double B[n * m], PB[n * m], G[m * n], Kt[m * n];
    double H[m * m], Rh[m * m];
    double p[n], w[n], c[n], xd[n], g[m], kt[m];
};

// acc[r][c] += sum_{q < len} X[q][x0 + r] * Y[q][y0 + c], X and Y row-major with leading dimensions
// ldx, ldy; x0, y0 even (16-byte aligned pairs).
template <int len>
__device__ __forceinline__ void tile_atb(const double* X, int ldx, int x0, const double* Y, int ldy, int y0,
                                         double (&acc)[2][2]) {
    double a2[2][2] = {{0.0, 0.0}, {0.0, 0.0}};      // second partial sums: halves the dependent chain
#pragma unroll
    for (int q = 0; q < len; ++q) {
        const double2 x = *reinterpret_cast<const double2*>(X + q * ldx + x0);
        const double2 y = *reinterpret_cast<const double2*>(Y + q * ldy + y0);
        if (q & 1) {
            a2[0][0] += x.x * y.x;  a2[0][1] += x.x * y.y;  a2[1][0] += x.y * y.x;  a2[1][1] += x.y * y.y;
        } else {
            acc[0][0] += x.x * y.x;  acc[0][1] += x.x * y.y;  acc[1][0] += x.y * y.x;  acc[1][1] += x.y * y.y;
        }
    }
    acc[0][0] += a2[0][0];  acc[0][1] += a2[0][1];  acc[1][0] += a2[1][0];  acc[1][1] += a2[1][1];
}
// acc[r][c] += sum_{q < len} X[x0 + r][q] * Y[q][y0 + c]   (rows of X, columns of Y; len even)
template <int len>
__device__ __forceinline__ void tile_ab(const double* X, int ldx, int x0, const double* Y, int ldy, int y0,
                                        double (&acc)[2][2]) {
    double a2[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
#pragma unroll
    for (int q = 0; q < len; q += 2) {
        const double2 x0v = *reinterpret_cast<const double2*>(X + (x0 + 0) * ldx + q);
        const double2 x1v = *reinterpret_cast<const double2*>(X + (x0 + 1) * ldx + q);
        const double2 ya = *reinterpret_cast<const double2*>(Y + q * ldy + y0);
        const double2 yb = *reinterpret_cast<const double2*>(Y + (q + 1) * ldy + y0);
        acc[0][0] += x0v.x * ya.x;  acc[0][1] += x0v.x * ya.y;  acc[1][0] += x1v.x * ya.x;  acc[1][1] += x1v.x * ya.y;
        a2[0][0] += x0v.y * yb.x;   a2[0][1] += x0v.y * yb.y;   a2[1][0] += x1v.y * yb.x;   a2[1][1] += x1v.y * yb.y;
    }
    acc[0][0] += a2[0][0];  acc[0][1] += a2[0][1];  acc[1][0] += a2[1][0];  acc[1][1] += a2[1][1];
}

template <int n, int m>
__global__ void __launch_bounds__(kTvlqrTiledThreads) tvlqr_riccati_tiled_kernel(const TvlqrArgs a) {
    static_assert(n % 2 == 0 && m % 2 == 0, "2 x 2 tiles");
    constexpr int G = kTvlqrTiledThreads;
    constexpr int hn = n / 2, hm = m / 2;
    static_assert(hn * hn <= 64 && hn * hm <= 32 && hm * hm <= 32 && n + 1 <= 32, "tile-to-warp mapping");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TvlqrTiledSmem<n, m>& s = *reinterpret_cast<TvlqrTiledSmem<n, m>*>(smem_raw);
    const int gt = threadIdx.x, warp = gt >> 5, lane = gt & 31;
    const int inst = blockIdx.x;
    const double* xd_i = a.xd + inst * a.xd_stride;
    const int t_hi = a.t_hi > 0 ? a.t_hi : a.T, t_lo = a.t_hi > 0 ? a.t_lo : 0;
    bool ok = true;
    // Work is assigned to warps by ROLE (one code path per warp and phase: no intra-warp divergence
    // between the tile kinds); tile origins are loop invariants.
    const int pa_r0 = 2 * (gt / hn), pa_c0 = 2 * (gt % hn);            // n x n tiles: threads 0 .. hn*hn-1
    const int pb_r0 = 2 * (lane / hm), pb_c0 = 2 * (lane % hm);        // n x m tiles: warp 2
    const int g_r0 = 2 * (lane / hn), g_c0 = 2 * (lane % hn);          // m x n tiles: warp 0
    const int h_r0 = 2 * (lane / hm), h_c0 = 2 * (lane % hm);          // m x m tiles: warp 1
    // running global pointers of step t (stepped back once per iteration: no 64-bit index math inside)
    constexpr int kRA = (n * n + G - 1) / G;
    const double* pA = a.At + ((long long)inst * a.T + (t_hi - 1)) * n * n + gt;
    const double* pB = a.Bt + ((long long)inst * a.T + (t_hi - 1)) * n * m + gt;
    const double* pc = a.ct + ((long long)inst * a.T + (t_hi - 1)) * n + gt;
    const double* pxd = xd_i + (long long)(t_hi - 1) * n + gt;
    double* pK = a.K + ((long long)inst * a.T + (t_hi - 1)) * m * n;
    double* pk = a.k + ((long long)inst * a.T + (t_hi - 1)) * m;
    static_assert(n * m <= G && n <= G, "one prefetch slot per thread for B, c, xd");
    double rA[kRA], rB = 0.0, rc = 0.0, rxd = 0.0;
    auto prefetch = [&] {
#pragma unroll
        for (int k = 0; k < kRA; ++k) if (gt + k * G < n * n) rA[k] = pA[k * G];
        if (gt < n * m) rB = *pB;
        if (gt < n) { rc = *pc;  rxd = *pxd; }
        pA -= n * n;  pB -= n * m;  pc -= n;  pxd -= n;
    };
    auto publish = [&] {
#pragma unroll
        for (int k = 0; k < kRA; ++k) if (gt + k * G < n * n) s.A[gt + k * G] = rA[k];
        if (gt < n * m) s.B[gt] = rB;
        if (gt < n) { s.c[gt] = rc;  s.xd[gt] = rxd; }
    };
    prefetch();
    // terminal condition: P_T = sym(Qd), p_T = -sym(Qd) xd_T (or the carried (P, p) of a later segment);
    // constants into shared memory, Q as sym(Q) (the weights' symmetric parts: see the generic kernel)
    double* carry_i = a.carry != nullptr ? a.carry + (long long)inst * (n * n + n) : nullptr;
    for (int e = gt; e < n * n; e += G) {
        const int i = e / n, j = e % n;
        s.P[e] = t_hi == a.T ? 0.5 * (a.Qd[e] + a.Qd[j * n + i]) : carry_i[e];
        s.Q[e] = 0.5 * (a.Q[e] + a.Q[j * n + i]);
    }
    for (int e = gt; e < m * m; e += G) s.Rh[e] = 0.5 * a.R[e];
    for (int i = gt; i < n; i += G) {
        if (t_hi == a.T) {
            double acc = 0.0;
            for (int q = 0; q < n; ++q) acc -= 0.5 * (a.Qd[i * n + q] + a.Qd[q * n + i]) * xd_i[(long long)a.T * n + q];
            s.p[i] = acc;
        } else {
            s.p[i] = carry_i[n * n + i];
        }
    }
    publish();
    __syncthreads();
    for (int t = t_hi - 1; t >= t_lo; --t) {
        if (t > t_lo) prefetch();
        // ---- phase 1: PA = P A (warps 0-1), PB = P B (warp 2), w = P c + p (warp 3) ----
        if (gt < hn * hn) {
            double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
            tile_ab<n>(s.P, n, pa_r0, s.A, n, pa_c0, acc);
            *reinterpret_cast<double2*>(&s.PA[pa_r0 * n + pa_c0]) = make_double2(acc[0][0], acc[0][1]);
            *reinterpret_cast<double2*>(&s.PA[(pa_r0 + 1) * n + pa_c0]) = make_double2(acc[1][0], acc[1][1]);
        } else if (warp == 2) {
            if (lane < hn * hm) {
                double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
                tile_ab<n>(s.P, n, pb_r0, s.B, m, pb_c0, acc);
                *reinterpret_cast<double2*>(&s.PB[pb_r0 * m + pb_c0]) = make_double2(acc[0][0], acc[0][1]);
                *reinterpret_cast<double2*>(&s.PB[(pb_r0 + 1) * m + pb_c0]) = make_double2(acc[1][0], acc[1][1]);
            }
        } else if (warp == 3) {
            if (lane < n) s.w[lane] = dot4<n>(&s.P[lane * n], 1, s.c, 1, s.p[lane]);
        }
        __syncthreads();
        // ---- phase 2: G = B' PA (warp 0), H = R/2 + B' PB (warp 1), g = B' w (warp 2) ----
        if (warp == 0) {
            if (lane < hm * hn) {
                double acc[2][2] = {{0.0, 0.0}, {0.0, 0.0}};
                tile_atb<n>(s.B, m, g_r0, s.PA, n, g_c0, acc);
                *reinterpret_cast<double2*>(&s.G[g_r0 * n + g_c0]) = make_double2(acc[0][0], acc[0][1]);
                *reinterpret_cast<double2*>(&s.G[(g_r0 + 1) * n + g_c0]) = make_double2(acc[1][0], acc[1][1]);
            }
        } else if (warp == 1) {
            if (lane < hm * hm) {
                double acc[2][2] = {{s.Rh[h_r0 * m + h_c0], s.Rh[h_r0 * m + h_c0 + 1]},
                                    {s.Rh[(h_r0 + 1) * m + h_c0], s.Rh[(h_r0 + 1) * m + h_c0 + 1]}};
                tile_atb<n>(s.B, m, h_r0, s.PB, m, h_c0, acc);
                *reinterpret_cast<double2*>(&s.H[h_r0 * m + h_c0]) = make_double2(acc[0][0], acc[0][1]);
                *reinterpret_cast<double2*>(&s.H[(h_r0 + 1) * m + h_c0]) = make_double2(acc[1][0], acc[1][1]);
            }
        } else if (warp == 2) {
            if (lane < m) s.g[lane] = dot4<n>(&s.B[lane], m, s.w, 1);
        }
        __syncthreads();
        // ---- phase 3: K = -H^-1 G, k = -H^-1 g (warp 0; H inverted redundantly in registers) ----
        if (gt <= n) {
            double Hs[m][m], Hi[m][m];
#pragma unroll
            for (int i = 0; i < m; ++i)
#pragma unroll
                for (int j = 0; j < m; ++j) Hs[i][j] = 0.5 * (s.H[i * m + j] + s.H[j * m + i]);
            ok = spd_inverse<m>(Hs, Hi) && ok;
            const int col = gt;
            double b[m], y[m];
#pragma unroll
            for (int i = 0; i < m; ++i) b[i] = col < n ? s.G[i * n + col] : s.g[i];
#pragma unroll
            for (int i = 0; i < m; ++i) {
                double acc = 0.0;
#pragma unroll
                for (int q = 0; q < m; ++q) acc -= Hi[i][q] * b[q];
                y[i] = acc;
            }
            if (col < n) {
#pragma unroll
                for (int i = 0; i < m; ++i) {
                    s.Kt[i * n + col] = y[i];
                    pK[i * n + col] = y[i];
                }
            } else {
#pragma unroll
                for (int i = 0; i < m; ++i) {
                    s.kt[i] = y[i];
                    pk[i] = y[i];
                }
            }
#pragma unroll
            for (int i = 0; i < m; ++i) ok = ok && isfinite(y[i]);
        }
        pK -= m * n;
        pk -= m;
        __syncthreads();
        // ---- phase 4: Pn = Q + A' PA + G' K (warps 0-1; raw, symmetrised when stored),
        //               p <- -sym(Q) xd_t + A' w + G' k (warp 2) ----
        double pnew = 0.0;
        if (gt < hn * hn) {
            double acc[2][2] = {{s.Q[pa_r0 * n + pa_c0], s.Q[pa_r0 * n + pa_c0 + 1]},
                                {s.Q[(pa_r0 + 1) * n + pa_c0], s.Q[(pa_r0 + 1) * n + pa_c0 + 1]}};
            tile_atb<n>(s.A, n, pa_r0, s.PA, n, pa_c0, acc);
            tile_atb<m>(s.G, n, pa_r0, s.Kt, n, pa_c0, acc);
            *reinterpret_cast<double2*>(&s.Pn[pa_r0 * n + pa_c0]) = make_double2(acc[0][0], acc[0][1]);
            *reinterpret_cast<double2*>(&s.Pn[(pa_r0 + 1) * n + pa_c0]) = make_double2(acc[1][0], acc[1][1]);
        } else if (warp == 2) {
            if (lane < n)
                pnew = (dot4<n>(&s.A[lane], n, s.w, 1) - dot4<n>(&s.Q[lane * n], 1, s.xd, 1)) +
                       dot4<m>(&s.G[lane], n, s.kt, 1);
        }
        __syncthreads();
        // ---- phase 5: P = sym(Pn), p, and the prefetched operands of step t-1 ----
        for (int e = gt; e < n * n; e += G) {
            const int i = e / n, j = e % n;
            s.P[e] = 0.5 * (s.Pn[i * n + j] + s.Pn[j * n + i]);
        }
        if (warp == 2 && lane < n) s.p[lane] = pnew;
        if (t > t_lo) publish();
        __syncthreads();
    }
    // NaN guard on the final value function (K_t, k_t: checked where written)
    for (int e = gt; e < n * n; e += G)
        if (!(s.P[e] == s.P[e])) ok = false;
    ok = __syncthreads_and(ok);
    // the first segment (from T) sets the status, later ones can only raise it
    if (gt == 0) a.status[inst] = (ok ? 0 : 1) | (t_hi == a.T ? 0 : a.status[inst]);
    if (t_lo > 0) {      // hand (P, p) of step t_lo to the next segment
        for (int e = gt; e < n * n; e += G) carry_i[e] = s.P[e];
        for (int i = gt; i < n; i += G) carry_i[n * n + i] = s.p[i];
    }
}

// ---------------------------------------------------------------------------------------------
// Throughput variant for MANY instances and n, m multiples of four (quadrotor 12/4; BASELINE.json
// configs[4]: 4096 instances).  The block kernel above is shared-memory bound there (73 % LSU, ~48 KB of
// operand traffic per instance and step with 2 x 2 tiles, a third of its threads busy, five block barriers
// per step).  Here TWO instances share a warp — 12 lanes each, lanes 24-31 retire at once — and every matrix
// product is cut into 4 x 4 register tiles of ONE code shape, so the lanes of both instances run the same
// instruction stream:
//     [PA | PB]          = P [A | B]                 12 x 16 -> 12 tiles, one per lane (P symmetric: rows = columns)
//     [A | B]^T [PA | PB], upper block triangle      6 tiles of A^T P A + 4 tiles of B^T [PA | PB] = [G | H0]
//     Pn (upper)        += G^T K                      6 tiles, 4 terms
// The lower block triangle of P is the mirror of the upper one (a lane stores its tile and its transpose; the
// diagonal tiles are symmetrised in registers), so the recursion keeps P exactly symmetric without a pass of
// its own.  The kernel is bound by the shared-memory pipe (one wavefront per clock and SM, an LDS.128 of a warp
// costs one per quarter warp with an active lane; ncu: profiles/r2_riccati_packed.txt), hence: the idle
// quarter warp exits, the second instance of a warp sits 16 bytes (mod 32) beside the first so that their
// quarter-warp-sharing lanes hit different banks, the rows of P [A | B], of P and of sym(Q) are shifted by 16 bytes
// per row group so that tile accesses of different row groups do too, and vector operands are read along contiguous rows (P is
// symmetric, and so is sym(Q)).  Eight instances per block of 128 threads, four blocks per SM: all 4096
// instances of configs[4] are resident at once.  Next step's operands are prefetched into registers (18
// doubles per lane) during the last product of the current step.
// ---------------------------------------------------------------------------------------------
constexpr int kRicPackThreads = 128;
constexpr int kRicPackLanes = 12;                       // lanes per instance
constexpr int kRicPackPerWarp = 2;                      // instances per warp
constexpr int kRicPackPerBlock = kRicPackPerWarp * kRicPackThreads / 32;
constexpr unsigned kRicPackMask = (1u << (kRicPackPerWarp * kRicPackLanes)) - 1u;      // the working lanes

template <int n, int m>
struct RicPackInst {
    static constexpr int W = n + m;
    static constexpr int kPab = n * W + 2 * (n / 4 - 1);      // rows of group g start 2 g doubles late
    static constexpr int kP = n * n + 2 * (n / 4 - 1);        // the same row-group shift for P (tile stores of the
                                                              // second product: three row groups in one quarter warp)
    double P[kP + (kP & 1)];      // value-function Hessian (exactly symmetric), row r at r n + 2 (r >> 2)
    double AB[n * W];             // [A | B] of the current step, row stride n + m
    double PAB[kPab + (kPab & 1)];  // P [A | B]
    double GH[m * W];             // B^T [PA | PB] = [G | H - R/2]
    double Kt[m * n];
    double p[n], w[n], c[n], xd[n], g[m], kt[m];
    double pad[2];                // size = 4 (mod 8) words: the warp's second instance lands on the other banks
    __device__ __forceinline__ static constexpr int pab_row(int r) { return r * W + 2 * (r >> 2); }
    __device__ __forceinline__ static constexpr int p_row(int r) { return r * n + 2 * (r >> 2); }
};
template <int n, int m>
struct RicPackSmem {
    double Qs[RicPackInst<n, m>::kP + (RicPackInst<n, m>::kP & 1)];      // sym(Q), rows shifted like P (tile loads)
    double Rh[m * m];                                                    // R / 2
    RicPackInst<n, m> inst[kRicPackPerBlock];
};

// acc[i][j] += sum_q X[q * ldx + x0 + i] * Y[row(q) + y0 + j]   (4 x 4 tile of X^T Y; x0, y0 multiples of 4);
// row(q) = q * ldy, plus the row-group shift of RicPackInst::PAB when YSHIFT (XSHIFT: the same for X = P)
template <int len, bool YSHIFT, bool XSHIFT = false>
__device__ __forceinline__ void tile4_atb(const double* X, int ldx, int x0, const double* Y, int ldy, int y0,
                                          double (&acc)[4][4]) {
    static_assert(len % 4 == 0, "row groups of four");
#pragma unroll 1      // one row group per trip: full unrolling hoists all 48 operand loads and spills at 128 registers
    for (int g = 0; g < len / 4; ++g) {
        const double* Xg = X + 4 * g * ldx + x0 + (XSHIFT ? 2 * g : 0);
        const double* Yg = Y + 4 * g * ldy + y0 + (YSHIFT ? 2 * g : 0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double2 xa = *reinterpret_cast<const double2*>(Xg + q * ldx);
            const double2 xb = *reinterpret_cast<const double2*>(Xg + q * ldx + 2);
            const double2 ya = *reinterpret_cast<const double2*>(Yg + q * ldy);
            const double2 yb = *reinterpret_cast<const double2*>(Yg + q * ldy + 2);
            const double x[4] = {xa.x, xa.y, xb.x, xb.y}, y[4] = {ya.x, ya.y, yb.x, yb.y};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fma(x[i], y[j], acc[i][j]);
        }
    }
}
// D[r0 + i][c0 + j] = acc[i][j] (TRANSPOSED: = acc[j][i]); `shift` doubles are added once (PAB row groups)
template <bool TRANSPOSED>
__device__ __forceinline__ void tile4_store(double* D, int ld, int r0, int c0, const double (&acc)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        double* d = D + (r0 + i) * ld + c0;
        if constexpr (TRANSPOSED) {
            *reinterpret_cast<double2*>(d) = make_double2(acc[0][i], acc[1][i]);
            *reinterpret_cast<double2*>(d + 2) = make_double2(acc[2][i], acc[3][i]);
        } else {
            *reinterpret_cast<double2*>(d) = make_double2(acc[i][0], acc[i][1]);
            *reinterpret_cast<double2*>(d + 2) = make_double2(acc[i][2], acc[i][3]);
        }
    }
}

template <int n, int m>
__global__ void __launch_bounds__(kRicPackThreads, 4) tvlqr_riccati_packed_kernel(const TvlqrArgs a) {
    static_assert(n == 12 && m == 4, "tile roles below are laid out for three row groups and one input group");
    using Inst = RicPackInst<n, m>;
    static_assert(sizeof(Inst) % 16 == 0 && (sizeof(Inst) / 4) % 8 == 4, "second instance of a warp: other banks");
    constexpr int W = n + m;                              // row stride of [A | B]
    constexpr int kOps = n * n + n * m + n + n;           // doubles of one step's operands: A, B, c, xd
    constexpr int kPre = (kOps + kRicPackLanes - 1) / kRicPackLanes;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    RicPackSmem<n, m>& sm = *reinterpret_cast<RicPackSmem<n, m>*>(smem_raw);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int e = tid; e < n * n; e += kRicPackThreads) {
        const int r = e / n, c = e % n;
        sm.Qs[Inst::p_row(r) + c] = 0.5 * (a.Q[e] + a.Q[c * n + r]);       // x' Q x only sees the symmetric part
    }
    for (int e = tid; e < m * m; e += kRicPackThreads) sm.Rh[e] = 0.5 * a.R[e];
    __syncthreads();
    if (lane >= kRicPackPerWarp * kRicPackLanes) return;   // the idle quarter warp: its loads would cost wavefronts
    const int sub = lane / kRicPackLanes;                 // instance of this lane inside the warp
    const int j = lane % kRicPackLanes;                   // role lane
    const int slot = warp * kRicPackPerWarp + sub;
    const long long inst_raw = (long long)blockIdx.x * kRicPackPerBlock + slot;
    // the lanes of a missing last instance shadow a valid one and write nothing outside their own slot
    const bool live = inst_raw < a.I;
    const long long inst = live ? inst_raw : (long long)a.I - 1;
    Inst& s = sm.inst[slot];
    const double* xd_i = a.xd + inst * a.xd_stride;
    const double* At = a.At + inst * a.T * n * n;
    const double* Bt = a.Bt + inst * a.T * n * m;
    const double* ct = a.ct + inst * a.T * n;
    // operand e of step t: A (n n) | B (n m) | c (n) | xd (n); lane j owns e = j, j + 12, ...
    double pre[kPre];
    auto prefetch = [&](int t) {
#pragma unroll
        for (int k = 0; k < kPre; ++k) {
            const int e = j + k * kRicPackLanes;
            if (e < n * n) pre[k] = At[(long long)t * n * n + e];
            else if (e < n * n + n * m) pre[k] = Bt[(long long)t * n * m + (e - n * n)];
            else if (e < n * n + n * m + n) pre[k] = ct[(long long)t * n + (e - n * n - n * m)];
            else if (e < kOps) pre[k] = xd_i[(long long)t * n + (e - n * n - n * m - n)];
        }
    };
    auto publish = [&] {
#pragma unroll
        for (int k = 0; k < kPre; ++k) {
            const int e = j + k * kRicPackLanes;
            if (e < n * n) s.AB[(e / n) * W + e % n] = pre[k];
            else if (e < n * n + n * m) s.AB[((e - n * n) / m) * W + n + (e - n * n) % m] = pre[k];
            else if (e < n * n + n * m + n) s.c[e - n * n - n * m] = pre[k];
            else if (e < kOps) s.xd[e - n * n - n * m - n] = pre[k];
        }
    };
    prefetch(a.T - 1);
    // terminal condition P_T = sym(Qd) (x' Qd x only sees the symmetric part), p_T = -sym(Qd) xd_T
    for (int e = j; e < n * n; e += kRicPackLanes) {
        const int r = e / n, c = e % n;
        s.P[Inst::p_row(r) + c] = 0.5 * (a.Qd[r * n + c] + a.Qd[c * n + r]);
    }
    {
        double acc = 0.0;
        for (int q = 0; q < n; ++q) acc -= 0.5 * (a.Qd[j * n + q] + a.Qd[q * n + j]) * xd_i[(long long)a.T * n + q];
        s.p[j] = acc;
    }
    publish();
    __syncwarp(kRicPackMask);
    bool ok = true;
    const int ab_r0 = 4 * (j / (W / 4)), ab_c0 = 4 * (j % (W / 4));      // tile of P [A | B]  (n/4 x W/4 tiles)
    // second product: lanes 0-5 the upper block triangle of A^T PA ((0,0) (0,4) (0,8) (4,4) (4,8) (8,8)),
    // lanes 6-9 the four tiles of B^T [PA | PB]
    const bool pn_tile = j < 6, gh_tile = j >= 6 && j < 6 + W / 4;
    const int pn_r0 = j < 3 ? 0 : (j < 5 ? 4 : 8);
    const int pn_c0 = j < 3 ? 4 * j : (j < 5 ? 4 * (j - 2) : 8);
    const int x0_2 = pn_tile ? pn_r0 : n;                                // columns of [A | B] that form X
    const int y0_2 = pn_tile ? pn_c0 : (gh_tile ? 4 * (j - 6) : 0);
    for (int t = a.T - 1; t >= 0; --t) {
        // ---- phase 1: [PA | PB] = P [A | B] (one 4 x 4 tile per lane), w = P c + p ----
        {
            double acc[4][4] = {};
            tile4_atb<n, false, true>(s.P, n, ab_r0, s.AB, W, ab_c0, acc);
            tile4_store<false>(s.PAB + 2 * (ab_r0 >> 2), W, ab_r0, ab_c0, acc);
            double wv = s.p[j];
#pragma unroll
            for (int q = 0; q < n; ++q) wv = fma(s.P[Inst::p_row(q) + j], s.c[q], wv);      // P[j][q] = P[q][j]
            s.w[j] = wv;
        }
        __syncwarp(kRicPackMask);
        // ---- phase 2: sym(Q) + A^T PA (upper block triangle, kept in registers) and [G | H0] = B^T [PA | PB];
        //               g = B^T w ----
        double pn[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int q = 0; q < 4; ++q) pn[i][q] = pn_tile ? sm.Qs[Inst::p_row(pn_r0 + i) + pn_c0 + q] : 0.0;
        if (pn_tile || gh_tile) {
            tile4_atb<n, true>(s.AB, W, x0_2, s.PAB, W, y0_2, pn);
            if (gh_tile) tile4_store<false>(s.GH, W, 0, y0_2, pn);
        }
        if (j < m) {
            double gv = 0.0;
#pragma unroll
            for (int q = 0; q < n; ++q) gv = fma(s.AB[q * W + n + j], s.w[q], gv);
            s.g[j] = gv;
        }
        __syncwarp(kRicPackMask);
        // ---- phase 3: K = -H^-1 G, k = -H^-1 g; column `j` (j = n: the affine term needs a 13th lane ->
        //      lane 0 does it after its own column); H = R/2 + sym(H0) inverted redundantly in registers ----
        {
            double Hs[m][m], Hi[m][m];
#pragma unroll
            for (int i = 0; i < m; ++i)
#pragma unroll
                for (int q = 0; q < m; ++q)
                    Hs[i][q] = 0.5 * ((s.GH[i * W + n + q] + sm.Rh[i * m + q]) + (s.GH[q * W + n + i] + sm.Rh[q * m + i]));
            ok = spd_inverse<m>(Hs, Hi) && ok;
            double* Kg = a.K + (inst * a.T + t) * m * n;
#pragma unroll
            for (int i = 0; i < m; ++i) {
                double acc = 0.0;
#pragma unroll
                for (int q = 0; q < m; ++q) acc = fma(-Hi[i][q], s.GH[q * W + j], acc);
                s.Kt[i * n + j] = acc;
                if (live) Kg[i * n + j] = acc;
                ok = ok && isfinite(acc);      // NaN / Inf in c or xd reach k only: checked below
            }
            if (j == 0) {
                double* kg = a.k + (inst * a.T + t) * m;
#pragma unroll
                for (int i = 0; i < m; ++i) {
                    double acc = 0.0;
#pragma unroll
                    for (int q = 0; q < m; ++q) acc = fma(-Hi[i][q], s.g[q], acc);
                    s.kt[i] = acc;
                    if (live) kg[i] = acc;
                    ok = ok && isfinite(acc);
                }
            }
        }
        __syncwarp(kRicPackMask);
        // next step's operands -> registers now (the 4 x 4 inverse of phase 3 is dead, the loads fly during
        // phase 4 and the other warps' work; prefetching a whole step ahead spilled at 128 registers)
        if (t > 0) prefetch(t - 1);
        // ---- phase 4: Pn += G^T K (lanes 0-5) -> P and its mirror (no phase reads P any more),
        //               p <- -sym(Q) xd_t + A^T w + G^T k (every lane one row; sym(Q) read along row j = column j) ----
        if (pn_tile) {
            tile4_atb<m, false>(s.GH, W, pn_r0, s.Kt, n, pn_c0, pn);
            if (pn_r0 == pn_c0) {
#pragma unroll
                for (int i = 1; i < 4; ++i)
#pragma unroll
                    for (int q = 0; q < i; ++q) pn[i][q] = pn[q][i] = 0.5 * (pn[i][q] + pn[q][i]);
            } else {
                tile4_store<true>(s.P + 2 * (pn_c0 >> 2), n, pn_c0, pn_r0, pn);
            }
            tile4_store<false>(s.P + 2 * (pn_r0 >> 2), n, pn_r0, pn_c0, pn);
        }
        double pnew;
        {
            double av = 0.0, qv = 0.0, gv = 0.0;
#pragma unroll
            for (int q = 0; q < n; ++q) {
                av = fma(s.AB[q * W + j], s.w[q], av);
                qv = fma(sm.Qs[Inst::p_row(q) + j], s.xd[q], qv);
            }
#pragma unroll
            for (int q = 0; q < m; ++q) gv = fma(s.GH[q * W + j], s.kt[q], gv);
            pnew = (av - qv) + gv;
        }
        __syncwarp(kRicPackMask);      // every read of [A | B], c, xd, p and w of this step is done
        s.p[j] = pnew;
        if (t > 0) publish();
        __syncwarp(kRicPackMask);
    }
    // NaN guard on the final value function (K_t, k_t: checked where written); one status per instance
    for (int e = j; e < n * n; e += kRicPackLanes) {
        const double v = s.P[Inst::p_row(e / n) + e % n];
        if (!(v == v)) ok = false;
    }
    ok = __all_sync(((1u << kRicPackLanes) - 1u) << (sub * kRicPackLanes), ok);
    if (live && j == 0) a.status[inst] = ok ? 0 : 1;
}

// ---------------------------------------------------------------------------------------------
// Rollouts (warp per instance; x lives in lane 0's registers).
//   closed loop: u_t = K_t x_t + k_t, x_{t+1} = f(x_t, u_t)      (irs_lqr.py:183-184)
//   open loop  : x_{t+1} = f(x_t, u_t) for given u               (irs_lqr.py:105-119)
// Both also return the cost of irs_lqr.py:121-137 (terminal term uses Q, :135-136).
// ---------------------------------------------------------------------------------------------
struct RolloutArgs {
    const double* K;      // [I, T, m, n] or nullptr (open loop)
    const double* k;      // [I, T, m]
    const double* x0;     // [I, n]
    const double* u_in;   // [I, T, m] (open loop)
    const double* xd;     // [I or 1, T+1, n]
    long long xd_stride;
    const double* Q;      // [n, n]
    const double* R;      // [m, m]
    double* x_trj;        // [I, T+1, n]
    double* u_trj;        // [I, T, m]
    double* cost;         // [I]
    int I, T;
    SysParams prm;
};

constexpr int kRolloutWarps = 2;

// IrsLqr.evaluate_cost (irs_lqr.py:121-137) of one instance by one warp, lanes over t; the terminal
// term uses Q (:135-136).  Returns the warp-reduced cost on every lane.
template <int n, int m>
__device__ __forceinline__ double warp_trajectory_cost(const double* x_trj, const double* u_trj,
                                                       const double* xd_i, const double* Q,
                                                       const double* R, int T, int lane) {
    double acc = 0.0;
    for (int t = lane; t <= T; t += 32) {
        // compiler barrier: without it the n*n + m*m loop-invariant weight loads below are hoisted out of
        // the t loop into registers (quadrotor: 160 doubles -> 255 registers and a 384-byte spill frame for
        // every kernel this routine is inlined into, the sequential rollouts among them)
        asm volatile("" ::: "memory");
        double e[n];
#pragma unroll
        for (int q = 0; q < n; ++q) e[q] = x_trj[(long long)t * n + q] - xd_i[(long long)t * n + q];
#pragma unroll
        for (int i = 0; i < n; ++i) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < n; ++q) s += Q[i * n + q] * e[q];
            acc += e[i] * s;
        }
        if (t < T) {
            double u[m];
#pragma unroll
            for (int q = 0; q < m; ++q) u[q] = u_trj[(long long)t * m + q];
#pragma unroll
            for (int i = 0; i < m; ++i) {
                double s = 0.0;
#pragma unroll
                for (int q = 0; q < m; ++q) s += R[i * m + q] * u[q];
                acc += u[i] * s;
            }
        }
    }
    return warp_sum(acc);
}

// One warp per instance.  The recursion x_{t+1} = f(x_t, u_t) is sequential and runs on lane 0 in
// fp64; the other lanes are the prefetcher: while lane 0 computes step t they fetch step t+1's
// gains / inputs into registers and hand them over through a double-buffered
// shared-memory slot, so the critical path never contains a global-memory round trip.
template <class Sys, bool CLOSED>
__global__ void __launch_bounds__(32 * kRolloutWarps) rollout_kernel(const RolloutArgs a) {
    constexpr int n = Sys::N, m = Sys::M;
    constexpr int kSlot = CLOSED ? m * n + m : m;        // K_t | k_t   or   u_t
    constexpr int kPer = (kSlot + 31) / 32;
    __shared__ double slot[kRolloutWarps][2][kSlot];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inst = blockIdx.x * kRolloutWarps + warp;
    if (inst >= a.I) return;
    const Sys sys(a.prm);
    const double* xd_i = a.xd + inst * a.xd_stride;
    double pre[kPer];
    auto fetch = [&](int t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int e = lane + 32 * k;
            if (e < kSlot) {
                if (CLOSED) pre[k] = e < m * n ? a.K[it * m * n + e] : a.k[it * m + (e - m * n)];
                else pre[k] = a.u_in[it * m + e];
            }
        }
    };
    auto publish = [&](int b) {
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int e = lane + 32 * k;
            if (e < kSlot) slot[warp][b][e] = pre[k];
        }
    };
    fetch(0);
    publish(0);
    __syncwarp();
    double x[n], u[m], xn[n];
    if (lane == 0) {
#pragma unroll
        for (int q = 0; q < n; ++q) {
            x[q] = a.x0[(long long)inst * n + q];
            a.x_trj[((long long)inst * (a.T + 1)) * n + q] = x[q];
        }
    }
    for (int t = 0; t < a.T; ++t) {
        const long long it = (long long)inst * a.T + t;
        const double* sl = slot[warp][t & 1];
        if (t + 1 < a.T) fetch(t + 1);                 // in flight while lane 0 computes
        if (lane == 0) {
            if (CLOSED) {
#pragma unroll
                for (int i = 0; i < m; ++i) {
                    double acc = sl[m * n + i];
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += sl[i * n + q] * x[q];
                    u[i] = acc;
                }
            } else {
#pragma unroll
                for (int i = 0; i < m; ++i) u[i] = sl[i];
            }
            sys.template step<false>(x, u, xn);
            if (CLOSED) {
#pragma unroll
                for (int i = 0; i < m; ++i) a.u_trj[it * m + i] = u[i];
            }
#pragma unroll
            for (int q = 0; q < n; ++q) {
                x[q] = xn[q];
                a.x_trj[((long long)inst * (a.T + 1) + t + 1) * n + q] = x[q];
            }
        }
        if (t + 1 < a.T) publish((t + 1) & 1);
        __syncwarp();
    }
    // cost of the finished trajectory, parallel over t (off the sequential path); lane 0's global
    // stores are visible to the warp after the __syncwarp that closed the loop
    __threadfence_block();
    __syncwarp();
    const double* u_used = CLOSED ? a.u_trj + (long long)inst * a.T * m : a.u_in + (long long)inst * a.T * m;
    const double c = warp_trajectory_cost<n, m>(a.x_trj + (long long)inst * (a.T + 1) * n, u_used, xd_i,
                                                a.Q, a.R, a.T, lane);
    if (lane == 0) a.cost[inst] = c;
}

// Rollout of LEARNED dynamics (systems.cuh: Mlp): one block of 128 threads per instance, thread j = hidden unit j
// with ITS rows of the first two layers in registers for the whole trajectory (the network does not change from
// step to step), the activations handed over through shared memory, two block barriers per layer.  The last layer
// runs on 4 n lanes: lane (k, c) carries partial chain c of output k.  Every unit is summed in exactly the order of
// Mlp::dot_row (four interleaved chains), so the trajectory is bit-identical to stepping the per-thread functor
// (test); a step costs ~0.3 us instead of the ~7 us of one warp reading the weights through L1 every step.
template <class Sys, bool CLOSED>
__global__ void __launch_bounds__(kMlpMaxHidden) rollout_mlp_kernel(const RolloutArgs a) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D, H = kMlpMaxHidden;
    static_assert(4 * n <= 32, "last layer: four chain lanes per output inside warp 0");
    __shared__ float in_s[d], a1_s[H], a2_s[H], out_s[n];
    const int tid = threadIdx.x, lane = tid & 31;
    const int inst = blockIdx.x;
    const Sys sys(a.prm);
    const MlpView& net = sys.net;
    const int H1 = net.H1, H2 = net.H2;
    const double* xd_i = a.xd + inst * a.xd_stride;
    // this thread's unit: first-layer row, hidden-layer row (zero weights beyond the widths: the products vanish
    // and the sums of the live units are unchanged)
    float w1r[d], b1r = 0.f, b2r = 0.f;
    float w2r[H];
#pragma unroll
    for (int q = 0; q < d; ++q) w1r[q] = tid < H1 ? __ldg(net.w1 + tid * d + q) : 0.f;
    if (tid < H1) b1r = __ldg(net.b1 + tid);
    if (tid < H2) b2r = __ldg(net.b2 + tid);
#pragma unroll
    for (int q = 0; q < H; ++q) w2r[q] = (tid < H2 && q < H1) ? __ldg(net.w2t + (long long)q * H2 + tid) : 0.f;
    // last layer: lane (k, c) of warp 0 holds w3[k][q] for q = c, c + 4, ... below the multiple of four, lane (k, 0)
    // also the tail q >= 4 (H2 / 4) — the order of dot_row
    const int ok = lane >> 2, oc = lane & 3;
    const int main4 = H2 & ~3;
    float w3r[H / 4], w3t[3];
#pragma unroll
    for (int i = 0; i < H / 4; ++i) w3r[i] = (tid < 4 * n && 4 * i + oc < main4) ? __ldg(net.w3 + (long long)ok * H2 + 4 * i + oc) : 0.f;
#pragma unroll
    for (int i = 0; i < 3; ++i) w3t[i] = (tid < 4 * n && oc == 0 && main4 + i < H2) ? __ldg(net.w3 + (long long)ok * H2 + main4 + i) : 0.f;
    const float b3r = (tid < 4 * n && oc == 0) ? __ldg(net.b3 + ok) : 0.f;

    double x[n], u[m];
#pragma unroll
    for (int q = 0; q < n; ++q) x[q] = a.x0[(long long)inst * n + q];
    if (tid == 0) {
#pragma unroll
        for (int q = 0; q < n; ++q) a.x_trj[((long long)inst * (a.T + 1)) * n + q] = x[q];
    }
    // gains / inputs of the NEXT step are loaded while the current one is evaluated (no global round trip on the
    // sequential path)
    constexpr int kGain = CLOSED ? m * n + m : m;
    double gain[kGain], gain_next[kGain];
    auto fetch = [&](int t, double (&g)[kGain]) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int e = 0; e < kGain; ++e) {
            if (CLOSED) g[e] = e < m * n ? a.K[it * m * n + e] : a.k[it * m + (e - m * n)];
            else g[e] = a.u_in[it * m + e];
        }
    };
    fetch(0, gain_next);
    for (int t = 0; t < a.T; ++t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int e = 0; e < kGain; ++e) gain[e] = gain_next[e];
        if (t + 1 < a.T) fetch(t + 1, gain_next);
        // every thread carries the state and forms the input (same operations on the same values)
        if (CLOSED) {
#pragma unroll
            for (int i = 0; i < m; ++i) {
                double acc = gain[m * n + i];
#pragma unroll
                for (int q = 0; q < n; ++q) acc += gain[i * n + q] * x[q];
                u[i] = acc;
            }
        } else {
#pragma unroll
            for (int i = 0; i < m; ++i) u[i] = gain[i];
        }
        float in[d];
#pragma unroll
        for (int q = 0; q < n; ++q) in[q] = (float)x[q];
#pragma unroll
        for (int q = 0; q < m; ++q) in[n + q] = (float)u[q];
        // layer 1 (as Mlp::hidden: sequential fmaf from the bias)
        {
            float sacc = b1r;
#pragma unroll
            for (int q = 0; q < d; ++q) sacc = fmaf(w1r[q], in[q], sacc);
            a1_s[tid] = tid < H1 ? fmaxf(sacc, 0.f) : 0.f;
        }
        __syncthreads();
        // layer 2 (as Mlp::dot_row with the transposed weights: chains q % 4 below the multiple of four, tail on chain 0)
        {
            float s0 = b2r, s1 = 0.f, s2 = 0.f, s3 = 0.f;
            const int m4 = H1 & ~3;
#pragma unroll
            for (int q = 0; q < H; q += 4) {
                if (q < m4) {
                    const float4 av = *reinterpret_cast<const float4*>(a1_s + q);
                    s0 = fmaf(w2r[q], av.x, s0);
                    s1 = fmaf(w2r[q + 1], av.y, s1);
                    s2 = fmaf(w2r[q + 2], av.z, s2);
                    s3 = fmaf(w2r[q + 3], av.w, s3);
                }
            }
#pragma unroll
            for (int q = 0; q < H; ++q)
                if (q >= m4 && q < H1) s0 = fmaf(w2r[q], a1_s[q], s0);
            a2_s[tid] = tid < H2 ? fmaxf((s0 + s1) + (s2 + s3), 0.f) : 0.f;
        }
        __syncthreads();
        // layer 3 on 4 n lanes of warp 0
        if (tid < 32) {
            float sc = b3r;
#pragma unroll
            for (int i = 0; i < H / 4; ++i)
                if (4 * i < main4) sc = fmaf(w3r[i], a2_s[4 * i + oc], sc);
#pragma unroll
            for (int i = 0; i < 3; ++i)
                if (main4 + i < H2) sc = fmaf(w3t[i], a2_s[main4 + i], sc);      // (zero weights off lane (k, 0))
            const float p1 = __shfl_down_sync(0xffffffffu, sc, 1);
            const float s01 = sc + p1;                        // lanes c = 0: s0 + s1; c = 2: s2 + s3
            const float p2 = __shfl_down_sync(0xffffffffu, s01, 2);
            if (tid < 4 * n && oc == 0) out_s[ok] = s01 + p2;  // (s0 + s1) + (s2 + s3)
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < n; ++q) x[q] = (double)out_s[q];
        if (tid == 0) {
            if (CLOSED) {
#pragma unroll
                for (int i = 0; i < m; ++i) a.u_trj[it * m + i] = u[i];
            }
#pragma unroll
            for (int q = 0; q < n; ++q) a.x_trj[((long long)inst * (a.T + 1) + t + 1) * n + q] = x[q];
        }
    }
    // cost of the finished trajectory by warp 0 (thread 0's stores: block-visible after the fence + barrier)
    __threadfence_block();
    __syncthreads();
    if (tid < 32) {
        const double* u_used = CLOSED ? a.u_trj + (long long)inst * a.T * m : a.u_in + (long long)inst * a.T * m;
        const double c = warp_trajectory_cost<n, m>(a.x_trj + (long long)inst * (a.T + 1) * n, u_used, xd_i, a.Q, a.R, a.T, lane);
        if (lane == 0) a.cost[inst] = c;
    }
}

// Rollout for systems whose next Euler angles do not depend on the input (Sys::kTrigAhead, the
// quadrotor): the three fp64 sincos evaluations are two thirds of a step on the sequential path, and
// the angles of step t+1 are known at the START of step t.  One block of two warps per instance:
// warp 0 carries the recursion exactly as rollout_kernel does (lane 0 computes, the other lanes
// prefetch the gains), warp 1 evaluates sin / cos of the next angles meanwhile (one lane per angle)
// and hands them over through a double-buffered shared slot; one block barrier per step.  Same
// operations on the same values as rollout_kernel (bit-identical, tests).
template <class Sys, bool CLOSED>
__global__ void __launch_bounds__(64) rollout_trig_kernel(const RolloutArgs a) {
    constexpr int n = Sys::N, m = Sys::M, kA = Sys::kTrigAhead;
    static_assert(kA > 0, "system has no input-independent angles");
    constexpr int kSlot = CLOSED ? m * n + m : m;        // K_t | k_t   or   u_t
    constexpr int kPer = (kSlot + 31) / 32;
    __shared__ double slot[2][kSlot];
    __shared__ double trig_s[2][2 * kA];                 // {sin, cos} of the angles of step t (buffer t & 1)
    __shared__ double angr_s[2][2 * kA];                 // angles | rates of the state x_t (buffer t & 1)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inst = blockIdx.x;
    const Sys sys(a.prm);
    const double* xd_i = a.xd + inst * a.xd_stride;
    double pre[kPer];
    auto fetch = [&](int t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int e = lane + 32 * k;
            if (e < kSlot) {
                if (CLOSED) pre[k] = e < m * n ? a.K[it * m * n + e] : a.k[it * m + (e - m * n)];
                else pre[k] = a.u_in[it * m + e];
            }
        }
    };
    auto publish = [&](int b) {
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int e = lane + 32 * k;
            if (e < kSlot) slot[b][e] = pre[k];
        }
    };
    double x[n], u[m], xn[n];
    if (warp == 0) {
        fetch(0);
        publish(0);
        if (lane == 0) {
#pragma unroll
            for (int q = 0; q < n; ++q) {
                x[q] = a.x0[(long long)inst * n + q];
                a.x_trj[((long long)inst * (a.T + 1)) * n + q] = x[q];
            }
#pragma unroll
            for (int j = 0; j < kA; ++j) { angr_s[0][j] = x[3 + j];  angr_s[0][kA + j] = x[9 + j]; }
        }
    } else if (lane < kA) {
        double sv, cv;
        Sys::trig(a.x0[(long long)inst * n + 3 + lane], sv, cv);
        trig_s[0][2 * lane] = sv;  trig_s[0][2 * lane + 1] = cv;
    }
    __syncthreads();
    for (int t = 0; t < a.T; ++t) {
        if (warp == 0) {
            const long long it = (long long)inst * a.T + t;
            const double* sl = slot[t & 1];
            if (t + 1 < a.T) fetch(t + 1);                 // in flight while lane 0 computes
            if (lane == 0) {
                if (CLOSED) {
#pragma unroll
                    for (int i = 0; i < m; ++i) {
                        double acc = sl[m * n + i];
#pragma unroll
                        for (int q = 0; q < n; ++q) acc += sl[i * n + q] * x[q];
                        u[i] = acc;
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < m; ++i) u[i] = sl[i];
                }
                double sc[2 * kA];
#pragma unroll
                for (int j = 0; j < 2 * kA; ++j) sc[j] = trig_s[t & 1][j];
                sys.template step_trig<false>(x, u, sc, xn);
                if (CLOSED) {
#pragma unroll
                    for (int i = 0; i < m; ++i) a.u_trj[it * m + i] = u[i];
                }
#pragma unroll
                for (int q = 0; q < n; ++q) {
                    x[q] = xn[q];
                    a.x_trj[((long long)inst * (a.T + 1) + t + 1) * n + q] = x[q];
                }
#pragma unroll
                for (int j = 0; j < kA; ++j) { angr_s[(t + 1) & 1][j] = x[3 + j];  angr_s[(t + 1) & 1][kA + j] = x[9 + j]; }
            }
            if (t + 1 < a.T) publish((t + 1) & 1);
        } else if (lane < kA && t + 1 < a.T) {
            // the angles of step t+1 from the state of step t (the expression of Sys::step itself)
            double sv, cv;
            Sys::trig(sys.next_angle(angr_s[t & 1][lane], angr_s[t & 1][kA + lane]), sv, cv);
            trig_s[(t + 1) & 1][2 * lane] = sv;  trig_s[(t + 1) & 1][2 * lane + 1] = cv;
        }
        __syncthreads();
    }
    // cost of the finished trajectory, parallel over t (off the sequential path)
    __threadfence_block();
    __syncthreads();
    if (warp == 0) {
        const double* u_used = CLOSED ? a.u_trj + (long long)inst * a.T * m : a.u_in + (long long)inst * a.T * m;
        const double c = warp_trajectory_cost<n, m>(a.x_trj + (long long)inst * (a.T + 1) * n, u_used, xd_i,
                                                    a.Q, a.R, a.T, lane);
        if (lane == 0) a.cost[inst] = c;
    }
}

// evaluate_cost for given trajectories (irs_lqr.py:121-137); one warp per instance, lanes over t.
template <int n, int m>
__global__ void __launch_bounds__(128) evaluate_cost_kernel(const double* x_trj, const double* u_trj,
                                                          const double* xd, long long xd_stride,
                                                          const double* Q, const double* R, int I, int T,
                                                          double* cost) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int inst = blockIdx.x * 4 + warp;
    if (inst >= I) return;
    const double* xd_i = xd + inst * xd_stride;
    const double acc = warp_trajectory_cost<n, m>(x_trj + (long long)inst * (T + 1) * n,
                                                  u_trj + (long long)inst * T * m, xd_i, Q, R, T, lane);
    if (lane == 0) cost[inst] = acc;
}

// Linear-model rollout for solve_tvlqr's return value (x*, u*) (tv_lqr.py:142-145):
// x_{t+1} = A_t x_t + B_t u_t + c_t with u_t = K_t x_t + k_t.
template <int n, int m>
__global__ void __launch_bounds__(64) linear_rollout_kernel(const TvlqrArgs a, const double* x0,
                                                           double* xs, double* us) {
    const int inst = blockIdx.x * blockDim.x + threadIdx.x;
    if (inst >= a.I) return;
    double x[n], u[m], xn[n];
#pragma unroll
    for (int q = 0; q < n; ++q) {
        x[q] = x0[(long long)inst * n + q];
        xs[((long long)inst * (a.T + 1)) * n + q] = x[q];
    }
    for (int t = 0; t < a.T; ++t) {
        const long long it = (long long)inst * a.T + t;
#pragma unroll
        for (int i = 0; i < m; ++i) {
            double acc = a.k[it * m + i];
#pragma unroll
            for (int q = 0; q < n; ++q) acc += a.K[(it * m + i) * n + q] * x[q];
            u[i] = acc;
            us[it * m + i] = acc;
        }
#pragma unroll
        for (int i = 0; i < n; ++i) {
            double acc = a.ct[it * n + i];
#pragma unroll
            for (int q = 0; q < n; ++q) acc += a.At[(it * n + i) * n + q] * x[q];
#pragma unroll
            for (int q = 0; q < m; ++q) acc += a.Bt[(it * n + i) * m + q] * u[q];
            xn[i] = acc;
        }
#pragma unroll
        for (int q = 0; q < n; ++q) {
            x[q] = xn[q];
            xs[((long long)inst * (a.T + 1) + t + 1) * n + q] = x[q];
        }
    }
}

}  // namespace irs
