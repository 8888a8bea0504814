// Box-constrained TVLQR (SURVEY.md section 8f row 1).
//
// The reference re-solves, at every timestep t0 of IrsLqr.local_descent (irs_lqr/irs_lqr.py:169-184),
// the QP of irs_lqr/tv_lqr.py:69-137 over the remaining horizon with absolute box bounds on states
// and inputs (:113-118, :132-134), and applies the first input to the true dynamics.
//
//   plan_check_kernel   for every start time t0 in parallel: roll the affine model forward from the
//                       ACTUAL state x_{t0} under the unconstrained gains and test the bounds.  If no
//                       plan touches a bound, every one of the reference's QPs had inactive
//                       constraints and the one-pass Riccati descent IS the reference's result.
//   box_mpc_kernel      otherwise: the reference's loop itself.  Each QP is solved by ADMM on the box
//                       split (y = z, y = states and inputs, z in the box); the equality-constrained
//                       step is an affine Riccati recursion whose MATRIX part (K_t, H_t^-1, P_t for
//                       the penalty-augmented cost) does not depend on the iterate nor on t0 and is
//                       computed once by tvlqr_riccati_kernel; only the vector recursion and the
//                       affine rollout run per iteration.  Consecutive QPs warm-start each other
//                       (split and dual variables are indexed by absolute time).
// Oracle: oracle/box_tvlqr.py (same algorithm in numpy, checked against a dense QP solve).
#pragma once
#include "tvlqr.cuh"

namespace irs {

struct PlanCheckArgs {
    const double* At;     // [I, T, n, n]
    const double* Bt;     // [I, T, n, m]
    const double* ct;     // [I, T, n]
    const double* K;      // [I, T, m, n]  unconstrained gains
    const double* k;      // [I, T, m]
    const double* x_trj;  // [I, T+1, n]   actual closed-loop states
    const double* xlo;    // [n]
    const double* xhi;
    const double* ulo;    // [m]
    const double* uhi;
    double tol;
    int* violated;        // [I] set to 1 if any plan leaves the box (zeroed by the entry point)
    double* scratch;      // [I, T, n+m, n+1]: closed-loop rows [A + B K | B k + c] and [K | k]
    int I, T;
};

// Stage 1, parallel over (t, instance): rows of the closed-loop map  x+ = (A + B K) x + (B k + c)  and
// of the feedback  u = K x + k, packed as (n + m) rows of n + 1 doubles.
template <int n, int m>
__global__ void __launch_bounds__(32) plan_rows_kernel(const PlanCheckArgs a) {
    constexpr int W = n + 1;
    const int lane = threadIdx.x;
    const int t = blockIdx.x, inst = blockIdx.y;
    const long long it = (long long)inst * a.T + t;
    double* out = a.scratch + it * (n + m) * W;
    for (int e = lane; e < (n + m) * W; e += 32) {
        const int r = e / W, c = e % W;
        double v;
        if (r < n) {
            const double* Br = a.Bt + (it * n + r) * m;
            if (c < n) {
                v = a.At[(it * n + r) * n + c];
#pragma unroll
                for (int q = 0; q < m; ++q) v += Br[q] * a.K[(it * m + q) * n + c];
            } else {
                v = a.ct[it * n + r];
#pragma unroll
                for (int q = 0; q < m; ++q) v += Br[q] * a.k[it * m + q];
            }
        } else {
            v = c < n ? a.K[(it * m + (r - n)) * n + c] : a.k[it * m + (r - n)];
        }
        out[e] = v;
    }
}

// Stage 2, grid = (T, I), one warp per (start time, instance): lanes 0..n-1 carry the planned state,
// lanes n..n+m-1 the planned input; one fused row product and one __syncwarp per step, next step's
// row prefetched into registers.
template <int n, int m>
__global__ void __launch_bounds__(32) plan_check_kernel(const PlanCheckArgs a) {
    static_assert(n + m <= 32, "one lane per coordinate");
    constexpr int W = n + 1;
    __shared__ double xs[2][n];
    const int lane = threadIdx.x;
    const int t0 = blockIdx.x, inst = blockIdx.y;
    const bool is_x = lane < n, active = lane < n + m;
    const double lo = !active ? 0.0 : (is_x ? a.xlo[lane] : a.ulo[lane - n]);
    const double hi = !active ? 0.0 : (is_x ? a.xhi[lane] : a.uhi[lane - n]);
    if (is_x) xs[0][lane] = a.x_trj[((long long)inst * (a.T + 1) + t0) * n + lane];
    const double* row = a.scratch + (((long long)inst * a.T + t0) * (n + m) + (active ? lane : 0)) * W;
    double r[W], rn[W];
#pragma unroll
    for (int q = 0; q < W; ++q) r[q] = row[q];
    __syncwarp();
    bool bad = false;
    int cur = 0;
    for (int t = t0; t < a.T; ++t) {
        if (t + 1 < a.T) {
#pragma unroll
            for (int q = 0; q < W; ++q) rn[q] = row[(long long)(n + m) * W + q];
            row += (long long)(n + m) * W;
        }
        double acc[4] = {r[n], 0.0, 0.0, 0.0};
#pragma unroll
        for (int q = 0; q < n; ++q) acc[q & 3] += r[q] * xs[cur][q];
        const double v = (acc[0] + acc[1]) + (acc[2] + acc[3]);
        if (active) bad |= !(v >= lo - a.tol && v <= hi + a.tol);
        if (is_x) xs[cur ^ 1][lane] = v;
        cur ^= 1;
#pragma unroll
        for (int q = 0; q < W; ++q) r[q] = rn[q];
        __syncwarp();
    }
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(&a.violated[inst], 1);
}

struct BoxMpcArgs {
    const double* At;     // [I, T, n, n]
    const double* Bt;     // [I, T, n, m]
    const double* ct;     // [I, T, n]
    const double* K;      // [I, T, m, n]   gains of the penalty-augmented problem
    const double* Hinv;   // [I, T, m, m]
    const double* P;      // [I, T+1, n, n]
    const double* Q;      // [n, n]  (original weights)
    const double* Qd;
    const double* R;      // [m, m]
    const double* xd;     // [I or 1, T+1, n]
    long long xd_stride;
    const double* dx;     // [n] ADMM penalties on the states
    const double* du;     // [m] ... on the inputs
    const double* xlo;    // [n], or [T+1, n] when xbox_stride = n (time-varying box, tv_lqr.py:113-114,:132-134)
    const double* xhi;
    const double* ulo;    // [m], or [T, m] when ubox_stride = m (tv_lqr.py:115-116)
    const double* uhi;
    long long xbox_stride, ubox_stride;      // 0: the box is constant over the horizon
    const double* x0;     // [I, n]
    const double* K0;     // [I, T, m, n]   unconstrained gains (or nullptr): a start time whose
    const double* k0;     // [I, T, m]      unconstrained plan stays inside the box skips its QP
    double tol;           // bound tolerance of that test
    double alpha, eps;
    int max_iter;
    int mpc;              // 1: closed loop on the true dynamics (local_descent); 0: one QP from x0 (solve_tvlqr)
    double* x_trj;        // [I, T+1, n]
    double* u_trj;        // [I, T, m]
    double* cost;         // [I] evaluate_cost of the result (irs_lqr.py:121-137)
    int* status;          // [I] 0 ok, 1 ADMM did not converge / NaN
    int* iters;           // [I] total ADMM iterations
    int I, T;
    SysParams prm;
};

// One warp per instance; lanes = coordinates.  Dynamic shared memory (doubles):
//   zx, wx, x : (T+1) n each     zu, wu, u, kk : T m each     Pc : T n     qxd : (T+1) n     scratch
//   CACHE: + the per-step matrices A_t, B_t, K_t, Hinv_t (and K0_t, k0_t), so that the sequential
//   sweeps read shared memory instead of chasing global-memory latency twice per step.
template <class Sys, bool CACHE>
__global__ void __launch_bounds__(32) box_mpc_kernel(const BoxMpcArgs a) {
    constexpr int n = Sys::N, m = Sys::M;
    static_assert(n <= 32 && m <= 32, "one lane per coordinate");
    extern __shared__ __align__(16) double sm[];
    const int T = a.T;
    double* zx = sm;
    double* wx = zx + (T + 1) * n;
    double* x = wx + (T + 1) * n;
    double* zu = x + (T + 1) * n;
    double* wu = zu + T * m;
    double* u = wu + T * m;
    double* kk = u + T * m;
    double* Pc = kk + T * m;
    double* qxd = Pc + T * n;     // sym(Q) xd_t (t < T), sym(Qd) xd_T
    double* pv = qxd + (T + 1) * n;   // [2][n] rolling p_{t+1}, p_t
    double* ww = pv + 2 * n;      // [n]
    double* gv = ww + n;          // [m]
    double* cache = gv + m;
    const int lane = threadIdx.x;
    const int inst = blockIdx.x;
    const long long base = (long long)inst * T;
    const double* xd_i = a.xd + inst * a.xd_stride;
    const Sys sys(a.prm);
    const double dxl = lane < n ? a.dx[lane] : 0.0, dul = lane < m ? a.du[lane] : 0.0;
    const bool can_skip = a.mpc && a.K0 != nullptr && a.k0 != nullptr;
    // per-step matrices: global (L1/L2) or staged in shared memory
    const double* Ap = a.At + base * n * n;
    const double* Bp = a.Bt + base * n * m;
    const double* Kp = a.K + base * m * n;
    const double* Hp = a.Hinv + base * m * m;
    const double* cp = a.ct + base * n;
    const double* K0p = can_skip ? a.K0 + base * m * n : nullptr;
    const double* k0p = can_skip ? a.k0 + base * m : nullptr;
    if constexpr (CACHE) {
        double* sA = cache;
        double* sB = sA + T * n * n;
        double* sK = sB + T * n * m;
        double* sH = sK + T * m * n;
        double* sc = sH + T * m * m;
        double* sK0 = sc + T * n;
        double* sk0 = sK0 + T * m * n;
        for (int e = lane; e < T * n * n; e += 32) sA[e] = Ap[e];
        for (int e = lane; e < T * n * m; e += 32) { sB[e] = Bp[e];  sK[e] = Kp[e]; }
        for (int e = lane; e < T * m * m; e += 32) sH[e] = Hp[e];
        for (int e = lane; e < T * n; e += 32) sc[e] = cp[e];
        if (can_skip) {
            for (int e = lane; e < T * m * n; e += 32) sK0[e] = K0p[e];
            for (int e = lane; e < T * m; e += 32) sk0[e] = k0p[e];
            K0p = sK0;  k0p = sk0;
        }
        Ap = sA;  Bp = sB;  Kp = sK;  Hp = sH;  cp = sc;
    }
    // Pc_t = P_{t+1} c_t, sym(Q) xd_t, sym(Qd) xd_T (the cost only sees the weights' symmetric parts, as
    // in tvlqr_riccati_kernel); cold start of the split variables: z = clip(target), w = 0
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
    int total_iters = 0;
    bool failed = false;
    const int n_starts = a.mpc ? T : 1;
    for (int t0 = 0; t0 < n_starts; ++t0) {
        bool solved = false;
        if (can_skip) {
            // unconstrained plan from the actual x_{t0}: if it stays inside the box the QP's bounds are
            // inactive and its first input is K0 x + k0 exactly (what the reference's solver returns)
            bool bad = false;
            for (int t = t0; t < T; ++t) {
                if (lane < m) {
                    double acc = k0p[t * m + lane];
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += K0p[(t * m + lane) * n + q] * x[t * n + q];
                    u[t * m + lane] = acc;
                    bad |= !(acc >= a.ulo[t * a.ubox_stride + lane] - a.tol && acc <= a.uhi[t * a.ubox_stride + lane] + a.tol);
                }
                __syncwarp();
                if (lane < n) {
                    double acc = cp[t * n + lane];
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += Ap[(t * n + lane) * n + q] * x[t * n + q];
#pragma unroll
                    for (int q = 0; q < m; ++q) acc += Bp[(t * n + lane) * m + q] * u[t * m + q];
                    x[(t + 1) * n + lane] = acc;
                    bad |= !(acc >= a.xlo[(t + 1) * a.xbox_stride + lane] - a.tol && acc <= a.xhi[(t + 1) * a.xbox_stride + lane] + a.tol);
                }
                __syncwarp();
                if (__any_sync(0xffffffffu, bad)) break;      // the ADMM recomputes the plan anyway
            }
            solved = !__any_sync(0xffffffffu, bad);
        }
        bool converged = solved;
        for (int it = 0; it < a.max_iter && !converged; ++it) {
            // ---- backward vector recursion: p_T, then kk_t, p_t for t = T-1 .. t0 ----
            int cur = 0;
            if (lane < n) pv[lane] = -(qxd[T * n + lane] + 0.5 * dxl * (zx[T * n + lane] - wx[T * n + lane]));
            __syncwarp();
            for (int t = T - 1; t >= t0; --t) {
                if (lane < n) ww[lane] = Pc[t * n + lane] + pv[cur * n + lane];
                __syncwarp();
                if (lane < m) {
                    double g = -0.5 * dul * (zu[t * m + lane] - wu[t * m + lane]);
                    const double* Bc = Bp + t * n * m + lane;
#pragma unroll
                    for (int q = 0; q < n; ++q) g += Bc[q * m] * ww[q];
                    gv[lane] = g;
                }
                __syncwarp();
                if (lane < m) {
                    const double* Hr = Hp + (t * m + lane) * m;
                    double acc = 0.0;
#pragma unroll
                    for (int q = 0; q < m; ++q) acc -= Hr[q] * gv[q];
                    kk[t * m + lane] = acc;
                }
                if (t > t0 && lane < n) {
                    double acc = -(qxd[t * n + lane] + 0.5 * dxl * (zx[t * n + lane] - wx[t * n + lane]));
                    const double* Ac = Ap + t * n * n + lane;
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += Ac[q * n] * ww[q];
                    const double* Kc = Kp + t * m * n + lane;
#pragma unroll
                    for (int q = 0; q < m; ++q) acc += Kc[q * n] * gv[q];
                    pv[(cur ^ 1) * n + lane] = acc;
                }
                cur ^= 1;
                __syncwarp();
            }
            // ---- forward affine rollout from the fixed x_{t0} ----
            for (int t = t0; t < T; ++t) {
                if (lane < m) {
                    const double* Kr = Kp + (t * m + lane) * n;
                    double acc = kk[t * m + lane];
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += Kr[q] * x[t * n + q];
                    u[t * m + lane] = acc;
                }
                __syncwarp();
                if (lane < n) {
                    const double* Ar = Ap + (t * n + lane) * n;
                    const double* Br = Bp + (t * n + lane) * m;
                    double acc = cp[t * n + lane];
#pragma unroll
                    for (int q = 0; q < n; ++q) acc += Ar[q] * x[t * n + q];
#pragma unroll
                    for (int q = 0; q < m; ++q) acc += Br[q] * u[t * m + q];
                    x[(t + 1) * n + lane] = acc;
                }
                __syncwarp();
            }
            // ---- relaxed projection, dual update, residuals (element-wise over the horizon) ----
            double r_prim = 0.0, r_dual = 0.0, scale = 1.0;
            for (int e = (t0 + 1) * n + lane; e < (T + 1) * n; e += 32) {
                const int i = e % n;
                const double xh = a.alpha * x[e] + (1.0 - a.alpha) * zx[e];
                const double zn = fmin(fmax(xh + wx[e], a.xlo[(e / n) * a.xbox_stride + i]), a.xhi[(e / n) * a.xbox_stride + i]);
                wx[e] += xh - zn;
                r_prim = fmax(r_prim, fabs(x[e] - zn));
                r_dual = fmax(r_dual, fabs(a.dx[i] * (zn - zx[e])));
                scale = fmax(scale, fabs(zn));
                zx[e] = zn;
            }
            for (int e = t0 * m + lane; e < T * m; e += 32) {
                const int j = e % m;
                const double uh = a.alpha * u[e] + (1.0 - a.alpha) * zu[e];
                const double zn = fmin(fmax(uh + wu[e], a.ulo[(e / m) * a.ubox_stride + j]), a.uhi[(e / m) * a.ubox_stride + j]);
                wu[e] += uh - zn;
                r_prim = fmax(r_prim, fabs(u[e] - zn));
                r_dual = fmax(r_dual, fabs(a.du[j] * (zn - zu[e])));
                scale = fmax(scale, fabs(zn));
                zu[e] = zn;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                r_prim = fmax(r_prim, __shfl_xor_sync(0xffffffffu, r_prim, o));
                r_dual = fmax(r_dual, __shfl_xor_sync(0xffffffffu, r_dual, o));
                scale = fmax(scale, __shfl_xor_sync(0xffffffffu, scale, o));
            }
            ++total_iters;
            // NaN-safe: a NaN residual never satisfies the test and the solve ends as "failed"
            converged = (r_prim <= a.eps * scale) && (r_dual <= a.eps * scale);
            __syncwarp();
        }
        if (!converged) failed = true;
        if (a.mpc) {
            // apply the first input (the feasible split variable; the unconstrained one if the QP was
            // skipped) to the TRUE dynamics (irs_lqr.py:183-184)
            if (lane == 0) {
                double xs[n], us[m], xn[n];
#pragma unroll
                for (int q = 0; q < n; ++q) xs[q] = x[t0 * n + q];
#pragma unroll
                for (int q = 0; q < m; ++q) us[q] = solved ? u[t0 * m + q] : zu[t0 * m + q];
                sys.template step<false>(xs, us, xn);
#pragma unroll
                for (int q = 0; q < n; ++q) x[(t0 + 1) * n + q] = xn[q];
#pragma unroll
                for (int q = 0; q < m; ++q) u[t0 * m + q] = us[q];
            }
            __syncwarp();
        }
    }
    // results: closed-loop trajectory (mpc) or the QP plan (states consistent with the dynamics)
    for (int e = lane; e < (T + 1) * n; e += 32) a.x_trj[(long long)inst * (T + 1) * n + e] = x[e];
    for (int e = lane; e < T * m; e += 32) a.u_trj[base * m + e] = u[e];
    __threadfence_block();
    __syncwarp();
    const double c = warp_trajectory_cost<n, m>(a.x_trj + (long long)inst * (T + 1) * n, a.u_trj + base * m, xd_i,
                                                a.Q, a.R, T, lane);
    if (lane == 0) {
        a.cost[inst] = c;
        a.status[inst] = (failed || !(c == c)) ? 1 : 0;
        a.iters[inst] = total_iters;
    }
}

template <int n, int m>
inline size_t box_mpc_smem_bytes(int T, bool cache) {
    size_t d = (size_t)3 * (T + 1) * n + (size_t)4 * T * m + (size_t)T * n + (size_t)(T + 1) * n + 2 * n + n + m;
    if (cache) d += (size_t)T * (n * n + 2 * n * m + m * m + n + m * n + m);
    return sizeof(double) * d;
}

}  // namespace irs
