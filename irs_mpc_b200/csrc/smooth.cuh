// Randomized-smoothing linearization kernels (SURVEY.md section 8, rows a12-a15).
//
//   smooth_zero_order_kernel<Sys,G>  fused: Philox noise (or replayed deltas) -> perturb ->
//                                    f(xbar+dx, ubar+du) -> delta f -> Gram accumulation of
//                                    [dx du]^T [dx du | delta f]  (irs_lqr_zero_order.py:49-57)
//   smooth_first_order_kernel<Sys>   same front end, accumulates the varying Jacobian scalars
//                                    (irs_lqr_first_order.py:42-48)
//   finalize_*_kernel                fixed-order fp64 reduction of the per-chunk partials,
//                                    Cholesky solve of the normal equations (== lstsq for full
//                                    column rank), c_t from the nominal point (:61-62)
#pragma once
#include "systems.cuh"

namespace irs {

enum SmoothFlags {
    kFlagSamplesBatchVariant = 1,   // samples use dynamics_batch semantics (irs_lqr_zero_order.py:51)
    kFlagProjectAbsolute = 2,       // three_cart_zero_order.py:43 quirk: sampling returns absolute points
    kFlagProjectDelta = 4,          // corrected variant: projected point minus nominal
    kFlagAntithetic = 8,            // Philox stream in antithetic pairs: sample 2q = +z_q, sample 2q+1 = -z_q
    kFlagCentered = 16,             // regressors are accumulated RELATIVE to the nominal point (xbar, ubar) together
                                    // with their first moments; the finalize undoes the shift in fp64 (implied by
                                    // kFlagProjectAbsolute; replayed absolute points: set explicitly)
};

struct SmoothArgs {
    const double* x_nom;   // [P, n] nominal states
    const double* u_nom;   // [P, m] nominal inputs
    const float* noise;    // [P, N, d] replayed deltas (dx | du) or nullptr
    float* partials;       // [P, C, NACC]
    long long N;           // samples per nominal point (local to this rank)
    long long S;           // samples per chunk
    int P, C;
    uint32_t seed_lo, seed_hi, iter, stream;
    uint32_t p0;           // global index of local point 0 (Philox counter word 1)
    unsigned long long i0; // global index of local sample 0 (Philox counter word 0)
    int flags;
    int nreg;              // n + m: live entries of sigma_scaled
    SysParams prm;
    float sigma_scaled[16];   // kBoxMullerScale * sigma[c] (Philox mode), lives in the constant bank
};
constexpr int kMaxRegressors = 16;

__host__ __device__ constexpr int gram_nacc(int n, int m) {
    return (n + m) * (n + m + 1) / 2 + (n + m) * n;
}
// Width of one packed partial block.  Systems whose regressors can be absolute points (three_cart's
// projection quirk, SURVEY Appendix A-5) append the first moments [sum z' (d) | sum dF (n)] of the
// centred accumulation (kFlagCentered); the entries are zero when a launch is not centred.
__host__ __device__ constexpr int gram_width(int n, int m, bool centered_capable) {
    return gram_nacc(n, m) + (centered_capable ? 2 * n + m : 0);
}
template <class Sys>
__host__ __device__ constexpr int gram_width_of() { return gram_width(Sys::N, Sys::M, Sys::kHasProjection); }
// packed upper-row layout: row i holds columns j = i..W-1, W = d + n
__host__ __device__ constexpr int gram_row_offset(int i, int W) { return i * W - i * (i - 1) / 2; }

// ---------------------------------------------------------------------------------------------
// One sample: regressors w[0..D) = (dx | du), responses w[D..D+N) = f(xbar+dx, ubar+du) - fbar.
// ---------------------------------------------------------------------------------------------
// w[c] = sigma[c] * normal_c of Philox counter (ctr0, point p, iteration, stream): ceil(d / 4) counter
// blocks, Box-Muller on word pairs (spec: oracle/philox_ref.py).
template <class Sys, int RS>
__device__ __forceinline__ void philox_normals(const SmoothArgs& a, int p, unsigned long long ctr0, float (&w)[RS]) {
    constexpr int d = Sys::D;
    constexpr int nblk = (d + 3) / 4;
#pragma unroll
    for (int j = 0; j < nblk; ++j) {
        uint32_t r[4];
        philox4x32((uint32_t)ctr0, a.p0 + (uint32_t)p, (a.iter << 8) | (uint32_t)j, a.stream,
                   a.seed_lo, a.seed_hi, r);
        float e[4];
        box_muller_raw(r[0], r[1], e[0], e[1]);
        box_muller_raw(r[2], r[3], e[2], e[3]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (4 * j + q < d) w[4 * j + q] = a.sigma_scaled[4 * j + q] * e[q];
    }
}

// Counter block j of philox_normals (w[4 j .. 4 j + 3]) for an antithetic pair evaluated in packed FP32
// (smooth_tc.cuh: kTcPaired): zz[q] = (w[4 j + q], w[4 j + q]), the bits of philox_normals in both halves of
// a register pair; Box-Muller and the sigma scaling run packed.  Entries past d are left unset.
template <class Sys>
__device__ __forceinline__ void philox_normals_x2(const SmoothArgs& a, int p, unsigned long long ctr0, int j,
                                                  float2 (&zz)[4]) {
    uint32_t r[4];
    philox4x32((uint32_t)ctr0, a.p0 + (uint32_t)p, (a.iter << 8) | (uint32_t)j, a.stream, a.seed_lo, a.seed_hi, r);
    float2 e01, e23;
    box_muller_raw_x2(r[0], r[1], r[2], r[3], e01, e23);
    const float e[4] = {e01.x, e01.y, e23.x, e23.y};
#pragma unroll
    for (int q = 0; q < 4; ++q)
        if (4 * j + q < Sys::D)
            zz[q] = Lanes<float2>::mul(Lanes<float2>::splat(a.sigma_scaled[4 * j + q]), Lanes<float2>::splat(e[q]));
}

// Deltas of sample i of nominal point p: replayed from a.noise or drawn from the Philox stream.
// MODE: -1 = decided at run time, 0 = Philox, 1 = replay (a compile-time mode keeps the test and the
// other path's code out of the hot loop).
template <class Sys, int RS, int MODE = -1>
__device__ __forceinline__ void draw_deltas(const SmoothArgs& a, int p, long long i, float (&w)[RS]) {
    constexpr int d = Sys::D;
    if (MODE == 1 || (MODE == -1 && a.noise != nullptr)) {
        const float* src = a.noise + ((long long)p * a.N + i) * d;
        if constexpr (d % 4 == 0) {
#pragma unroll
            for (int c = 0; c < d; c += 4) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(src + c));
                w[c] = v.x;  w[c + 1] = v.y;  w[c + 2] = v.z;  w[c + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int c = 0; c < d; ++c) w[c] = __ldg(src + c);
        }
    } else {
        unsigned long long gi = a.i0 + (unsigned long long)i;
        if (a.flags & kFlagAntithetic) {
            // antithetic pairs: samples 2q and 2q + 1 are +z_q and -z_q, one Philox draw per PAIR
            const bool minus = (gi & 1ull) != 0;
            philox_normals<Sys, RS>(a, p, gi >> 1, w);
            if (minus) {
#pragma unroll
                for (int c = 0; c < d; ++c) w[c] = -w[c];
            }
        } else {
            philox_normals<Sys, RS>(a, p, gi, w);
        }
    }
}

// three_cart: project the perturbed state onto non-penetration
// (three_cart_dynamics.py:196-264 called from three_cart_zero_order.py:38-43).
// The POSITIONS are projected in fp64: the reference re-evaluates its masks on the partially
// projected point, and after a pair push-out the gap it re-tests is exactly d in exact arithmetic,
// so whether the next push-out (which has a real depth) fires is decided by the rounding of the
// reference's float64 operations; only the same arithmetic on the same values reproduces those
// decisions.  Everything that no branch depends on (velocities, inputs) stays in fp32.
// pos64: the kProj leading nominal coordinates in fp64 (shared memory), or nullptr = read a.x_nom.
//
// In BOTH projection modes w leaves this function RELATIVE to the nominal point:
//     w[c] = fl32(proj(xbar + dx)[c] - xbar[c])  for the projected coordinates, w unchanged otherwise.
// kFlagProjectDelta: that IS the regressor and the perturbation.  kFlagProjectAbsolute — the
// reference closure returns ABSOLUTE points, which the solver adds to the nominal AGAIN and uses
// un-centred as regressors (SURVEY Appendix A-5), reproduced literally: the state handed to the
// dynamics is xbar + (xbar + w) (the callers perturb the doubled nominal, systems.cuh: centred_frame) and
// the regressors are xbar + w, accumulated as w with their first moments and shifted back in fp64 by
// the finalize (kFlagCentered).  An fp32 Gram of the absolute points themselves loses the sample spread once
// |xbar| >> sigma, which the quirk's meaningless linearization reaches after one descent.
template <class Sys, int RS>
__device__ __forceinline__ void project_deltas(const SmoothArgs& a, int p, const double* pos64, float (&w)[RS]) {
    constexpr int n = Sys::N;
    if constexpr (Sys::kHasProjection) {
        constexpr int kProj = Sys::kProjDims;
        if (a.flags & (kFlagProjectAbsolute | kFlagProjectDelta)) {
            using SysD = typename Sys::template Rebind<double>;
            const SysD sysd(a.prm);
            double xb[kProj], xp[n];
#pragma unroll
            for (int c = 0; c < kProj; ++c) {
                xb[c] = pos64 != nullptr ? pos64[c] : a.x_nom[(long long)p * n + c];
                xp[c] = xb[c] + (double)w[c];
            }
#pragma unroll
            for (int c = kProj; c < n; ++c) xp[c] = 0.0;      // untouched by project()
            sysd.project(xp);
#pragma unroll
            for (int c = 0; c < kProj; ++c) w[c] = (float)(xp[c] - xb[c]);
        }
    }
}

// Replayed regressors that are absolute points (kFlagCentered without an in-kernel projection):
// w[c] <- fl32(w[c] - nominal[c]) with the fp64 nominal, AFTER the state has been formed.
template <class Sys, int RS>
__device__ __forceinline__ void center_replayed(const SmoothArgs& a, int p, float (&w)[RS]) {
    constexpr int n = Sys::N, m = Sys::M;
#pragma unroll
    for (int c = 0; c < n; ++c) w[c] = (float)((double)w[c] - a.x_nom[(long long)p * n + c]);
#pragma unroll
    for (int c = 0; c < m; ++c) w[n + c] = (float)((double)w[n + c] - a.u_nom[(long long)p * m + c]);
}

template <class Sys, bool BATCH, int RS>
__device__ __forceinline__ void make_sample(const Sys& sys, const SmoothArgs& a, int p, long long i,
                                            const float* xbar, const float* ubar,
                                            const float* fbar, float (&w)[RS], bool want_df = true) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    draw_deltas<Sys, RS>(a, p, i, w);
    project_deltas<Sys, RS>(a, p, nullptr, w);
    if constexpr (Sys::kHasProjection) {
        // replayed absolute points -> relative to the nominal (the caller's xbar is then the centred frame)
        if ((a.flags & kFlagCentered) && !(a.flags & kFlagProjectAbsolute)) center_replayed<Sys, RS>(a, p, w);
    }
    float x[n], u[m];
#pragma unroll
    for (int c = 0; c < n; ++c) x[c] = xbar[c] + w[c];
#pragma unroll
    for (int c = 0; c < m; ++c) u[c] = ubar[c] + w[n + c];
    if (want_df) {
        float f[n];
        sys.template step<BATCH>(x, u, f);
#pragma unroll
        for (int c = 0; c < n; ++c) w[d + c] = f[c] - fbar[c];
    } else {
        // first-order path: hand the perturbed point back in place of the responses
#pragma unroll
        for (int c = 0; c < n; ++c) w[c] = x[c];
#pragma unroll
        for (int c = 0; c < m; ++c) w[n + c] = u[c];
    }
}

// Row ownership when the Gram rows are split over G warps: rows are paired (i, D-1-i) so that
// every pair carries the same number of outputs; pair q belongs to warp q % G.
__host__ __device__ constexpr bool owns_row(int i, int D, int G, int g) {
    return ((i < D - 1 - i ? i : D - 1 - i) % G) == g;
}
__host__ __device__ constexpr int role_pairs(int D, int Wp, int G, int g) {
    int k = 0;
    for (int i = 0; i < D; ++i)
        if (owns_row(i, D, G, g)) k += Wp / 2 - i / 2;
    return k;
}
// smem row stride (floats): multiple of 4 with an odd number of 16-byte units -> the 8 lanes of a
// quarter warp reading consecutive rows with LDS.128 hit 8 distinct bank groups.
__host__ __device__ constexpr int smem_row_stride(int Wp) {
    int rs = (Wp + 3) / 4 * 4;
    if ((rs / 4) % 2 == 0) rs += 4;
    return rs;
}

template <class Sys, int G>
struct ZeroOrderCfg {
    static constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    static constexpr int W = d + n;
    static constexpr int Wp = (W + 1) / 2 * 2;
    static constexpr int RS = G == 1 ? Wp : smem_row_stride(Wp);
    static constexpr int NACC = gram_nacc(n, m);
    static constexpr int kThreads = 32 * (G == 1 ? 4 : G);
    static constexpr int kTile = 32 * G;             // samples per round when G > 1
};

// Accumulate role g's share of the Gram update for one sample row w (registers).
template <class Sys, int G, int g, int NP>
__device__ __forceinline__ void gram_update(const float* w, float2 (&acc)[NP]) {
    using C = ZeroOrderCfg<Sys, G>;
    int k = 0;
#pragma unroll
    for (int i = 0; i < C::d; ++i) {
        if (owns_row(i, C::d, G, g)) {
            const float2 zi = make_float2(w[i], w[i]);
#pragma unroll
            for (int jj = i / 2; jj < C::Wp / 2; ++jj) {
                acc[k] = ffma2(zi, make_float2(w[2 * jj], w[2 * jj + 1]), acc[k]);
                ++k;
            }
        }
    }
}

// Warp-reduce role g's accumulators and write them into the packed partial block.
template <class Sys, int G, int g, int NP>
__device__ __forceinline__ void gram_flush(float2 (&acc)[NP], float* out, int lane) {
    using C = ZeroOrderCfg<Sys, G>;
    int k = 0;
#pragma unroll
    for (int i = 0; i < C::d; ++i) {
        if (owns_row(i, C::d, G, g)) {
#pragma unroll
            for (int jj = i / 2; jj < C::Wp / 2; ++jj) {
                const float sx = warp_sum(acc[k].x);
                const float sy = warp_sum(acc[k].y);
                ++k;
                if (lane == 0) {
                    const int j0 = 2 * jj, j1 = 2 * jj + 1;
                    if (j0 >= i && j0 < C::W) out[gram_row_offset(i, C::W) + j0 - i] = sx;
                    if (j1 >= i && j1 < C::W) out[gram_row_offset(i, C::W) + j1 - i] = sy;
                }
            }
        }
    }
}

// Role g's share of the Gram update for the G*32 samples of one smem tile (lane = sample).
template <class Sys, int G, int g, int NP>
__device__ __forceinline__ void gram_update_tile(const float* tile, int lane, float2 (&acc)[NP]) {
    using C = ZeroOrderCfg<Sys, G>;
#pragma unroll 1
    for (int q = 0; q < G; ++q) {
        float w[C::RS];
        const float4* src = reinterpret_cast<const float4*>(tile + (q * 32 + lane) * C::RS);
#pragma unroll
        for (int c = 0; c < C::RS / 4; ++c) {
            const float4 v = src[c];
            w[4 * c] = v.x;  w[4 * c + 1] = v.y;  w[4 * c + 2] = v.z;  w[4 * c + 3] = v.w;
        }
        gram_update<Sys, G, g, NP>(w, acc);
    }
}

// G == 1: every thread keeps the whole Gram block of its own samples in registers.
template <class Sys, bool BATCH>
__device__ __forceinline__ void zero_order_registers(const Sys& sys, const SmoothArgs& a, int p,
                                                     long long s_begin, long long s_end,
                                                     const float* xbar, const float* ubar,
                                                     const float* fbar, float* slabs, float* out) {
    using C = ZeroOrderCfg<Sys, 1>;
    constexpr int NP = role_pairs(C::d, C::Wp, 1, 0);
    constexpr int WIDTH = gram_width_of<Sys>();
    constexpr int NMOM = WIDTH - C::NACC;                    // first moments (centred-capable systems)
    float2 acc[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) acc[k] = make_float2(0.f, 0.f);
    float mom[NMOM > 0 ? NMOM : 1];
#pragma unroll
    for (int k = 0; k < (NMOM > 0 ? NMOM : 1); ++k) mom[k] = 0.f;
    const int lane = threadIdx.x & 31;
    for (long long s = s_begin + threadIdx.x; s < s_end; s += C::kThreads) {
        float w[C::RS];
#pragma unroll
        for (int c = 0; c < C::RS; ++c) w[c] = 0.f;
        make_sample<Sys, BATCH, C::RS>(sys, a, p, s, xbar, ubar, fbar, w);
        gram_update<Sys, 1, 0, NP>(w, acc);
        if constexpr (NMOM > 0) {
#pragma unroll
            for (int k = 0; k < NMOM; ++k) mom[k] += w[k];
        }
    }
    // cross-warp: each warp flushes into its own smem slab, then the block sums the slabs
    float* slab = slabs + (threadIdx.x >> 5) * WIDTH;
    gram_flush<Sys, 1, 0, NP>(acc, slab, lane);
    if constexpr (NMOM > 0) {
#pragma unroll
        for (int k = 0; k < NMOM; ++k) {
            const float v = warp_sum(mom[k]);
            if (lane == 0) slab[C::NACC + k] = (a.flags & (kFlagCentered | kFlagProjectAbsolute)) ? v : 0.f;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < WIDTH; e += C::kThreads) {
        float s = 0.f;
#pragma unroll
        for (int wq = 0; wq < C::kThreads / 32; ++wq) s += slabs[wq * WIDTH + e];
        out[e] = s;
    }
}

// G > 1: the Gram rows are split over the G warps of the block.  Sample generation is COMMON code
// (one copy in the instruction stream); only the short accumulate/flush sections are specialised
// per warp role, so the hot loop stays inside the instruction cache.  The sample tile is double
// buffered: one __syncthreads per round.
template <class Sys, int G>
__device__ __forceinline__ void zero_order_split(const Sys& sys, const SmoothArgs& a, int p,
                                                 long long s_begin, long long s_end,
                                                 const float* xbar, const float* ubar,
                                                 const float* fbar, float* tiles, float* out) {
    using C = ZeroOrderCfg<Sys, G>;
    constexpr int NP = role_pairs(C::d, C::Wp, G, 0);
    static_assert(G == 4, "supported group size");
    static_assert(role_pairs(C::d, C::Wp, G, G - 1) == NP && role_pairs(C::d, C::Wp, G, 1) == NP,
                  "row split must be balanced");
    float2 acc[NP];
#pragma unroll
    for (int k = 0; k < NP; ++k) acc[k] = make_float2(0.f, 0.f);
    const int lane = threadIdx.x & 31;
    const int role = threadIdx.x >> 5;
    int buf = 0;
    for (long long base = s_begin; base < s_end; base += C::kTile) {
        float* tile = tiles + buf * (C::kTile * C::RS);
        {
            float w[C::RS];
#pragma unroll
            for (int c = 0; c < C::RS; ++c) w[c] = 0.f;
            const long long s = base + threadIdx.x;
            if (s < s_end) make_sample<Sys, false, C::RS>(sys, a, p, s, xbar, ubar, fbar, w);
            float4* dst = reinterpret_cast<float4*>(tile + threadIdx.x * C::RS);
#pragma unroll
            for (int c = 0; c < C::RS / 4; ++c)
                dst[c] = make_float4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
        }
        __syncthreads();
        switch (role) {
            case 0: gram_update_tile<Sys, G, 0, NP>(tile, lane, acc); break;
            case 1: gram_update_tile<Sys, G, 1, NP>(tile, lane, acc); break;
            case 2: gram_update_tile<Sys, G, 2 % G, NP>(tile, lane, acc); break;
            default: gram_update_tile<Sys, G, 3 % G, NP>(tile, lane, acc); break;
        }
        buf ^= 1;
    }
    switch (role) {
        case 0: gram_flush<Sys, G, 0, NP>(acc, out, lane); break;
        case 1: gram_flush<Sys, G, 1, NP>(acc, out, lane); break;
        case 2: gram_flush<Sys, G, 2 % G, NP>(acc, out, lane); break;
        default: gram_flush<Sys, G, 3 % G, NP>(acc, out, lane); break;
    }
}

template <class Sys, int G>
__global__ void __launch_bounds__(ZeroOrderCfg<Sys, G>::kThreads, G == 1 ? 1 : 3)
smooth_zero_order_kernel(const SmoothArgs a) {
    constexpr int n = Sys::N, m = Sys::M;
    extern __shared__ __align__(16) float tile[];
    const Sys sys(a.prm);
    const int p = blockIdx.x / a.C;
    const int c = blockIdx.x % a.C;
    const long long s_begin = (long long)c * a.S;
    const long long s_end = s_begin + a.S < a.N ? s_begin + a.S : a.N;
    float xbar[n], ubar[m], fbar[n];
#pragma unroll
    for (int q = 0; q < n; ++q) xbar[q] = (float)a.x_nom[(long long)p * n + q];
#pragma unroll
    for (int q = 0; q < m; ++q) ubar[q] = (float)a.u_nom[(long long)p * m + q];
    // nominal response: the reference uses the SCALAR dynamics here (irs_lqr_zero_order.py:52); a centred
    // accumulation measures against the sample dynamics at the doubled nominal (smooth_tc.cuh:
    // reference_response; the finalize adds the difference back in fp64)
    bool centred = false;
    if constexpr (Sys::kHasProjection) centred = (a.flags & (kFlagCentered | kFlagProjectAbsolute)) != 0;
    if (centred) {
        double xd[n], ud[m];
#pragma unroll
        for (int q = 0; q < n; ++q) xd[q] = a.x_nom[(long long)p * n + q];
#pragma unroll
        for (int q = 0; q < m; ++q) ud[q] = a.u_nom[(long long)p * m + q];
        centred_frame<Sys>(xd, ud, xbar, ubar);       // the samples are perturbed around the centred frame
        if (a.flags & kFlagSamplesBatchVariant) sys.template step<true>(xbar, ubar, fbar);
        else sys.template step<false>(xbar, ubar, fbar);
    } else {
        sys.template step<false>(xbar, ubar, fbar);
    }
    float* out = a.partials + ((long long)p * a.C + c) * gram_width_of<Sys>();
    if constexpr (G == 1) {
        if (a.flags & kFlagSamplesBatchVariant)
            zero_order_registers<Sys, true>(sys, a, p, s_begin, s_end, xbar, ubar, fbar, tile, out);
        else
            zero_order_registers<Sys, false>(sys, a, p, s_begin, s_end, xbar, ubar, fbar, tile, out);
    } else {
        // the split path is only instantiated for systems whose batch and scalar dynamics agree
        static_assert(!Sys::kHasProjection, "split path assumes step<true> == step<false>");
        zero_order_split<Sys, G>(sys, a, p, s_begin, s_end, xbar, ubar, fbar, tile, out);
    }
}

// ---------------------------------------------------------------------------------------------
// First-order: accumulate the NJ varying Jacobian scalars (irs_lqr_first_order.py:42-48).
// partials layout [P, C, NJ].
// ---------------------------------------------------------------------------------------------
template <class Sys>
__global__ void __launch_bounds__(128) smooth_first_order_kernel(const SmoothArgs a) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    constexpr int NJ = Sys::NJ > 0 ? Sys::NJ : 1;
    constexpr int RS = d + n;
    __shared__ float slab[4][NJ];
    const Sys sys(a.prm);
    const int p = blockIdx.x / a.C;
    const int c = blockIdx.x % a.C;
    const long long s_begin = (long long)c * a.S;
    const long long s_end = s_begin + a.S < a.N ? s_begin + a.S : a.N;
    float xbar[n], ubar[m], fbar[n];
#pragma unroll
    for (int q = 0; q < n; ++q) xbar[q] = (float)a.x_nom[(long long)p * n + q];
#pragma unroll
    for (int q = 0; q < m; ++q) ubar[q] = (float)a.u_nom[(long long)p * m + q];
#pragma unroll
    for (int q = 0; q < n; ++q) fbar[q] = 0.f;
    float acc[NJ];
#pragma unroll
    for (int k = 0; k < NJ; ++k) acc[k] = 0.f;
    for (long long s = s_begin + threadIdx.x; s < s_end; s += 128) {
        float w[RS];
        make_sample<Sys, false, RS>(sys, a, p, s, xbar, ubar, fbar, w, /*want_df=*/false);
        float v[NJ];
        sys.jac_var(w, w + n, v);
#pragma unroll
        for (int k = 0; k < NJ; ++k) acc[k] += v[k];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NJ; ++k) {
        const float s = warp_sum(acc[k]);
        if (lane == 0) slab[warp][k] = s;
    }
    __syncthreads();
    float* out = a.partials + ((long long)p * a.C + c) * NJ;
    for (int k = threadIdx.x; k < NJ; k += 128) out[k] = (slab[0][k] + slab[1][k]) + (slab[2][k] + slab[3][k]);
}

// ---------------------------------------------------------------------------------------------
// Finalize (fp64).  Few points: one block of 128 threads per nominal point (latency: the sum over
// chunks and the nominal dynamics run beside the warp that factors the Gram).  Many points: four
// threads per point (finalize_zero_order_quad_kernel below).
// ---------------------------------------------------------------------------------------------
constexpr int kFinalizeThreads = 128;

// Index tables of the finalize kernel, one per system, built at COMPILE time (constant-initialised
// __device__ data: present on every device of the process without an upload, no host-side state):
// packed Gram entry e -> (i, j), packed lower-triangle entry -> (row, col).  (A per-block search for
// them costs more than the factorisation itself when a block owns a single point.)
constexpr int kMaxGramEntries = kMaxRegressors * (kMaxRegressors + 1) / 2 + kMaxRegressors * kMaxRegressors;
constexpr int kMaxTriEntries = kMaxRegressors * (kMaxRegressors + 1) / 2;
struct FinalizeTables {
    unsigned char gram_i[kMaxGramEntries], gram_j[kMaxGramEntries];
    unsigned char tri_r[kMaxTriEntries], tri_c[kMaxTriEntries];
};
constexpr FinalizeTables make_finalize_tables(int n, int m) {
    FinalizeTables t{};
    const int d = n + m, W = d + n;
    int e = 0;
    for (int i = 0; i < d; ++i)
        for (int j = i; j < W; ++j, ++e) { t.gram_i[e] = (unsigned char)i;  t.gram_j[e] = (unsigned char)j; }
    e = 0;
    for (int r = 0; r < d; ++r)
        for (int c = 0; c <= r; ++c, ++e) { t.tri_r[e] = (unsigned char)r;  t.tri_c[e] = (unsigned char)c; }
    return t;
}
// indexed by SystemId: pendulum, bicycle, quadrotor, three_cart, learned 2/1 (, the user system)
__device__ const FinalizeTables g_finalize_tables[kNumSystems] = {
    make_finalize_tables(2, 1), make_finalize_tables(5, 2), make_finalize_tables(12, 4), make_finalize_tables(6, 2),
#ifdef IRS_USER_SYSTEM
    make_finalize_tables(2, 1), make_finalize_tables(IRS_USER_N, IRS_USER_M)};
#else
    make_finalize_tables(2, 1)};
#endif

// Fused sample-sharded exchange (one process per GPU, peer-mapped buffers over NVLink): see
// peer_exchange_point below.  world == 0: not sharded.
struct PeerFusedArgs {
    double* const* peer_bufs;     // [world] device array: base of each rank's exchange buffer
    int* const* peer_flags;       // [world] device array: base of each rank's flag array [world][flag_stride]
    int* epoch;                   // local: exchanges completed so far (advanced by the last block of a launch)
    unsigned int* done_counter;   // local: blocks of the current launch that have finished (reset by the last)
    long long slot_stride;        // doubles per (parity, rank) slot (>= P * width)
    int flag_stride;              // flags per rank row (>= P)
    int rank, world;
    unsigned long long timeout_ns;
    // mode kPeerGather (timestep-sharded run): peer_bufs are the ranks' OUTPUT buffers
    // [2 parities][At: P_total n n | Bt: P_total n m | ct: P_total n | status: P_total] doubles
    // (out_stride doubles per parity), peer_flags their flag arrays [P_total]; this rank owns the global
    // points p0 .. p0 + P - 1
    int mode;
    int p0, P_total;
    long long out_stride;
};
enum PeerMode { kPeerNone = 0, kPeerExchange = 1, kPeerGather = 2 };

struct FinalizeArgs {
    const double* x_nom;     // [P, n]
    const double* u_nom;     // [P, m]
    const float* partials;   // [R][P, C, width] fp32 per-chunk partials (width = NACC or NJ), or
    const double* reduced;   // [R][P, width] fp64 chunk-reduced sums (exactly one of the two is set)
    long long rank_stride;   // elements between rank buffers (R buffers are summed in rank order)
    int R;
    int P, C;
    double n_total;          // total samples per point (first order: divisor of the mean)
    double* At;              // [P, n, n]
    double* Bt;              // [P, n, m]
    double* ct;              // [P, n]
    int* status;             // [P] 0 ok, 1 rank-deficient Gram
    const FinalizeTables* tables;   // index tables of this system (device)
    int centered;                   // the Gram was accumulated relative to the nominal point: undo the shift
    PeerFusedArgs peer;             // fused exchange of the sample-sharded path (world == 0: unused)
    SysParams prm;
};

// Where a finalize block reads its sums from: the launch arguments, or (fused exchange) the local
// exchange buffer of the current epoch.
struct PartialSource {
    const float* partials;
    const double* reduced;
    long long rank_stride;
    int R, C;
};
__device__ __forceinline__ PartialSource partial_source(const FinalizeArgs& a) {
    return PartialSource{a.partials, a.reduced, a.rank_stride, a.R, a.C};
}

// Fixed-order sum over ranks, then chunks, of entry e of point p (deterministic; the chunk loop is
// unrolled by eight so that the loads are in flight together while the adds keep their order).
__device__ __forceinline__ double sum_partials(const PartialSource& a, int p, int e, int width) {
    double s = 0.0;
    if (a.reduced != nullptr) {
        // rank blocks (L2: may be peer-written): eight loads in flight, adds in rank order — one load latency per
        // eight ranks instead of one per rank (8 GPUs: 32 serial L2 round trips per thread of the fused exchange)
        const double* src = a.reduced + (long long)p * width + e;
        int r = 0;
        for (; r + 8 <= a.R; r += 8) {
            double v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = __ldcg(src + (long long)(r + k) * a.rank_stride);
#pragma unroll
            for (int k = 0; k < 8; ++k) s += v[k];
        }
        if (r + 4 <= a.R) {
            double v[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) v[k] = __ldcg(src + (long long)(r + k) * a.rank_stride);
#pragma unroll
            for (int k = 0; k < 4; ++k) s += v[k];
            r += 4;
        }
        for (; r < a.R; ++r) s += __ldcg(src + (long long)r * a.rank_stride);
        return s;
    }
    for (int r = 0; r < a.R; ++r) {
        const float* src = a.partials + r * a.rank_stride + ((long long)p * a.C) * width + e;
        int c = 0;
        for (; c + 8 <= a.C; c += 8) {       // eight loads in flight, adds in chunk order
            float v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = src[(long long)(c + k) * width];
#pragma unroll
            for (int k = 0; k < 8; ++k) s += (double)v[k];
        }
        for (; c < a.C; ++c) s += (double)src[(long long)c * width];
    }
    return s;
}

// sum_{c < C} src[c * width] in chunk order, eight loads in flight (the adds keep their order).
__device__ __forceinline__ double sum_chunks_in_order(const float* src, int C, int width) {
    double s = 0.0;
    int c = 0;
    for (; c + 8 <= C; c += 8) {
        float v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = src[(long long)(c + k) * width];
#pragma unroll
        for (int k = 0; k < 8; ++k) s += (double)v[k];
    }
    for (; c < C; ++c) s += (double)src[(long long)c * width];
    return s;
}

// ---------------------------------------------------------------------------------------------
// Sample-sharded exchange FUSED into the finalize kernel (one process per GPU, peer-mapped exchange
// buffers over NVLink / NVSwitch; torch symmetric memory provides the address exchange only).
// The block that owns nominal point p
//   1. reduces its rank's fp32 per-chunk partials of p to fp64 (fixed chunk order) and stores each
//      value straight into slot `rank` of EVERY rank's exchange buffer (NVLink stores),
//   2. raises this rank's arrival flag of point p on every rank (system-scope release), and
//   3. waits (acquire loads, timeout instead of a hang) until every rank's block of p has arrived,
// after which the ordinary finalize sums the `world` blocks in rank order from the LOCAL buffer.
// No separate reduction / wait kernels, no NCCL call: compute, all-gather and fit are one launch,
// and a point is fitted as soon as ITS blocks are there, not when the whole step is.
// Flags carry the exchange epoch (never reset; the epoch lives in device memory and is advanced by
// the last block of a launch, so the sequence is CUDA-graph replayable and a changed grid — a
// shorter horizon — cannot desynchronise it); buffers are double buffered by epoch parity: a rank
// can run at most one exchange ahead of a peer, because its next kernel needs that peer's next flags.
// Blocks only ever wait for REMOTE blocks of the same point, so the launch needs all its blocks
// co-resident on every rank (the host checks P against the occupancy and uses NCCL beyond that).
// Returns the epoch; *timed_out = a peer did not deliver in time (the caller flags status 2).
// ---------------------------------------------------------------------------------------------
template <int BT>
__device__ __forceinline__ int peer_exchange_point(const FinalizeArgs& a, int p, int width, int tid,
                                                   PartialSource* src, bool* timed_out) {
    const PeerFusedArgs& x = a.peer;
    // every block reads the epoch before the LAST block of this launch advances it
    const int epoch = *reinterpret_cast<volatile int*>(x.epoch) + 1;
    const long long slot0 = (long long)(epoch & 1) * x.world * x.slot_stride;
    const long long mine = slot0 + (long long)x.rank * x.slot_stride + (long long)p * width;
    for (int e = tid; e < width; e += BT) {
        const double s = sum_chunks_in_order(a.partials + ((long long)p * a.C) * width + e, a.C, width);
        for (int r = 0; r < x.world; ++r) x.peer_bufs[r][mine + e] = s;      // local for r == rank
    }
    // the barrier orders the block's stores before the flag threads, whose system-scope RELEASE stores are
    // cumulative: `world` fences per block instead of one per thread (each is a MEMBAR.SYS + L1 invalidate)
    __syncthreads();
    int late = 0;
    if (tid < x.world) {
        int* remote = x.peer_flags[tid] + (long long)x.rank * x.flag_stride + p;
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(remote), "r"(epoch) : "memory");
        const int* local = x.peer_flags[x.rank] + (long long)tid * x.flag_stride + p;
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        // relaxed polls, ONE acquire fence once the flag is there (an acquire load per poll is a MEMBAR.SYS and an L1
        // invalidate each time round)
        while (true) {
            int v;
            asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(local) : "memory");
            if (v >= epoch) break;
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > x.timeout_ns) { late = 1;  break; }
            __nanosleep(100);
        }
        asm volatile("fence.acq_rel.sys;" ::: "memory");
    }
    *timed_out = __syncthreads_or(late) != 0;
    src->partials = nullptr;
    src->reduced = x.peer_bufs[x.rank] + slot0;
    src->rank_stride = x.slot_stride;
    src->R = x.world;
    src->C = 1;
    return epoch;
}

// Last block of a fused launch: reset the block counter and publish the epoch (all other blocks have
// finished, hence read the old epoch already).
__device__ __forceinline__ void peer_exchange_finish(const FinalizeArgs& a, int epoch, int tid) {
    __syncthreads();
    if (tid == 0) {
        const unsigned int ticket = atomicAdd(a.peer.done_counter, 1u) + 1u;
        if (ticket == gridDim.x) {
            *a.peer.done_counter = 0u;
            __threadfence();
            *reinterpret_cast<volatile int*>(a.peer.epoch) = epoch;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Timestep-sharded run: the all-gather of the per-step blocks [A_t | B_t | c_t] FUSED into the finalize
// kernel.  The block of local point p writes its result straight into EVERY rank's output buffer at the
// global point index (NVLink stores; 205 doubles per quadrotor step and rank) and raises that point's
// arrival flag on every rank; the LAST block of the launch then waits until the flags of all P_total
// points have arrived here, so when the kernel completes the full linearization is in local memory —
// no NCCL call, no packing kernels, and nothing for a consumer to wait on.  Only the last block waits,
// and only for remote blocks, which never wait for this rank: no co-residency requirement.  Epoch in
// device memory, output double buffered by epoch parity (as for the sample-sharded exchange): a rank
// can be one step ahead of a peer, never two.
// ---------------------------------------------------------------------------------------------
template <class Sys, int BT>
__device__ __forceinline__ void write_abc_gather(const FinalizeArgs& a, int p, const double* AB,
                                                 const double* nom /*[n+m+n] smem*/, int status_value,
                                                 int epoch, int tid) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    const PeerFusedArgs& x = a.peer;
    const long long g = (long long)x.p0 + p, Pt = x.P_total;
    const long long slot = (long long)(epoch & 1) * x.out_stride;
    double cval = 0.0;
    if (tid < n) {
        cval = nom[d + tid];
#pragma unroll
        for (int q = 0; q < d; ++q) cval = fma(-AB[tid * d + q], nom[q], cval);
    }
    for (int r = 0; r < x.world; ++r) {
        double* At = x.peer_bufs[r] + slot;
        double* Bt = At + Pt * n * n;
        double* ct = Bt + Pt * n * m;
        double* st = ct + Pt * n;
        for (int e = tid; e < n * d; e += BT) {
            const int row = e / d, cidx = e % d;
            if (cidx < n) At[(g * n + row) * n + cidx] = AB[e];
            else Bt[(g * n + row) * m + (cidx - n)] = AB[e];
        }
        if (tid < n) ct[g * n + tid] = cval;
        if (tid == 0) st[g] = (double)status_value;
    }
    __syncthreads();      // (cumulative release stores below: see peer_exchange_point)
    if (tid < x.world) {
        int* remote = x.peer_flags[tid] + g;
        asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(remote), "r"(epoch) : "memory");
    }
}

// Last block of a gather launch (or the only block of a rank without points): wait for all points.
template <int BT>
__device__ __forceinline__ void peer_gather_wait(const PeerFusedArgs& x, int epoch, int tid) {
    const int* local = x.peer_flags[x.rank];
    double* st = x.peer_bufs[x.rank] + (long long)(epoch & 1) * x.out_stride + x.out_stride - x.P_total;
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (int g = tid; g < x.P_total; g += BT) {
        while (true) {
            int v;
            asm volatile("ld.relaxed.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(local + g) : "memory");
            if (v >= epoch) break;
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (t - t0 > x.timeout_ns) { st[g] = 2.0;  break; }      // status 2: the point never arrived
            __nanosleep(100);
        }
    }
    asm volatile("fence.acq_rel.sys;" ::: "memory");      // one acquire after the relaxed polls
    __syncthreads();
    if (tid == 0) {
        *x.done_counter = 0u;
        __threadfence();
        *reinterpret_cast<volatile int*>(x.epoch) = epoch;
    }
}

template <int BT>
__device__ __forceinline__ void peer_gather_finish(const FinalizeArgs& a, int epoch, int tid) {
    __shared__ bool last_block;
    __syncthreads();
    if (tid == 0) last_block = atomicAdd(a.peer.done_counter, 1u) + 1u == gridDim.x;
    __syncthreads();
    if (last_block) peer_gather_wait<BT>(a.peer, epoch, tid);
}

// A rank that owns no timestep of a gather step still takes part in it (epochs stay in step).
__global__ void __launch_bounds__(128) peer_gather_wait_kernel(const PeerFusedArgs x) {
    const int epoch = *reinterpret_cast<volatile int*>(x.epoch) + 1;
    peer_gather_wait<128>(x, epoch, threadIdx.x);
}

// Compile-time loop: f(std::integral_constant<int, I>) for I = I0 .. I1 - 1 (the triangular loop
// nests must be unrolled at compile time so that the solution stays in registers).
template <int I0, int I1, class F>
__device__ __forceinline__ void static_for(F&& f) {
    if constexpr (I0 < I1) {
        f(std::integral_constant<int, I0>{});
        static_for<I0 + 1, I1>(f);
    }
}

// Fixed-order sums (ranks, then chunks: the order of sum_partials) of U entries of one point at once;
// the loads of the U entries are independent, so they are in flight together.  CB > 1: the loads of CB
// chunks are issued before the first of their adds as well (one L2 round trip per CB chunks instead of
// one per chunk; the adds keep their order, so the sums do not depend on CB).  CB * U floats of registers;
// CB > 1 has a block barrier between the loads and the adds: every thread of the block must call it.
// pbase = offset of the point inside a rank buffer (chunk 0), rel[u] = entry index, < 0 = none (sum 0).
template <int U, int CB = 1>
__device__ __forceinline__ void sum_partials_multi(const PartialSource& a, long long pbase, const int (&rel)[U],
                                                   int width, double (&s)[U]) {
#pragma unroll
    for (int u = 0; u < U; ++u) s[u] = 0.0;
    for (int r = 0; r < a.R; ++r) {
        if (a.reduced != nullptr) {
            const double* src = a.reduced + r * a.rank_stride + pbase;
            double v[U];
#pragma unroll
            for (int u = 0; u < U; ++u) v[u] = rel[u] >= 0 ? __ldcg(src + rel[u]) : 0.0;      // L2: may be peer-written
#pragma unroll
            for (int u = 0; u < U; ++u) s[u] += v[u];
        } else {
            const float* src = a.partials + r * a.rank_stride + pbase;
            for (int c = 0; c < a.C; c += CB, src += CB * width) {
                float v[CB][U];
#pragma unroll
                for (int k = 0; k < CB; ++k) {
                    // past the last chunk: load the last one again and drop it (a branch around the load would
                    // let the compiler convert each value right after its load, i.e. wait for it)
                    const int kk = c + k < a.C ? k : a.C - 1 - c;
#pragma unroll
                    for (int u = 0; u < U; ++u) v[k][u] = rel[u] >= 0 ? src[kk * width + rel[u]] : 0.f;
                }
                // Fence: without it the compiler interleaves the adds with the loads, and the first add to
                // wait for its load holds back every load behind it.  A barrier alone does not stop that (the
                // conversions are register work and move above it), so every value is OR-ed with the
                // barrier's result, which is 0 (C >= 1): the adds now depend on the barrier, the loads stay
                // above it, and the bits are untouched.  tools/finalize_phases.py reports the schedule.
                if constexpr (CB > 1) {
                    const int zero = __syncthreads_or(a.C < 1);
#pragma unroll
                    for (int k = 0; k < CB; ++k)
#pragma unroll
                        for (int u = 0; u < U; ++u) v[k][u] = __int_as_float(__float_as_int(v[k][u]) | zero);
                }
#pragma unroll
                for (int k = 0; k < CB; ++k)
                    if (c + k < a.C) {
#pragma unroll
                        for (int u = 0; u < U; ++u) s[u] += (double)v[k][u];
                    }
            }
        }
    }
}

// Nominal point (xbar | ubar | f(xbar, ubar)) of point p in fp64 -> shared memory.  f(xbar, ubar)
// (scalar dynamics, …zero_order.py:61) was written into ct[p] by the dynamics kernel that
// irs_smooth_finalize launches first in the many-points case, which keeps the fp64 dynamics (and its
// ~250 registers) out of the throughput variant of this kernel.
template <class Sys, int BT>
__device__ __forceinline__ void nominal_to_smem(const FinalizeArgs& a, int p, double* nom, int tid) {
    constexpr int n = Sys::N, m = Sys::M;
    for (int q = tid; q < 2 * n + m; q += BT) {
        nom[q] = q < n ? a.x_nom[(long long)p * n + q]
                       : (q < n + m ? a.u_nom[(long long)p * m + (q - n)] : a.ct[(long long)p * n + (q - n - m)]);
    }
}

// Latency variant: one thread evaluates f(xbar, ubar) in fp64 itself (it runs on warp 1 while warp 0
// factors the Gram), which saves the separate dynamics launch when there are only a few points.
template <class Sys>
__device__ __forceinline__ void nominal_compute_to_smem(const FinalizeArgs& a, int p, double* nom) {
    constexpr int n = Sys::N, m = Sys::M;
    const Sys sys(a.prm);
    double xb[n], ub[m], fb[n];
#pragma unroll
    for (int q = 0; q < n; ++q) xb[q] = a.x_nom[(long long)p * n + q];
#pragma unroll
    for (int q = 0; q < m; ++q) ub[q] = a.u_nom[(long long)p * m + q];
    sys.template step<false>(xb, ub, fb);      // scalar dynamics at the nominal (…zero_order.py:61)
#pragma unroll
    for (int q = 0; q < n; ++q) nom[q] = xb[q];
#pragma unroll
    for (int q = 0; q < m; ++q) nom[n + q] = ub[q];
#pragma unroll
    for (int q = 0; q < n; ++q) nom[n + m + q] = fb[q];
}

// At, Bt from AB ([n][d] smem) and c = f(xbar,ubar) - A xbar - B ubar (…zero_order.py:59-62).
template <class Sys, int BT>
__device__ __forceinline__ void write_abc(const FinalizeArgs& a, int p, const double* AB,
                                          const double* nom /*[n+m+n] smem*/, int tid) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    for (int e = tid; e < n * d; e += BT) {
        const int r = e / d, cidx = e % d;
        if (cidx < n) a.At[((long long)p * n + r) * n + cidx] = AB[e];
        else a.Bt[((long long)p * n + r) * m + (cidx - n)] = AB[e];
    }
    if (tid < n) {
        double acc = nom[d + tid];
#pragma unroll
        for (int q = 0; q < d; ++q) acc = fma(-AB[tid * d + q], nom[q], acc);
        a.ct[(long long)p * n + tid] = acc;
    }
}

// Chunks whose loads a thread of finalize_zero_order_kernel has in flight at once (<= 3 entries per
// thread: 96 floats of registers): a point's partials cost ceil(C / 32) L2 round trips instead of C
// (C = 25 at N = 1e5: one).
constexpr int kFinalizeChunksInFlight = 32;

// Phase clock of finalize_zero_order_kernel (tools/finalize_phases.py builds the library with
// -DIRS_FINALIZE_PHASES; the shipped library has no stamps): SM clock and global timer at each phase
// boundary of block 0, read back through irs_finalize_phases().
#ifdef IRS_FINALIZE_PHASES
enum FinalizePhase { kPhStart, kPhSums, kPhGram, kPhNominal, kPhFactor, kPhSolve, kPhWritten, kNumFinalizePhases };
__device__ unsigned long long g_finalize_phases[2 * kNumFinalizePhases];
// Every lane of the warp runs the stamp and the stores are predicated: a branch would leave the warp
// diverged after it, and the shuffles of the factorisation would then take their slow path.
__device__ __forceinline__ void finalize_stamp(int k, bool on) {
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    const unsigned long long clk = (unsigned long long)clock64();
    asm volatile("{ .reg .pred p;  setp.ne.u32 p, %0, 0;  @p st.global.u64 [%1], %2;  @p st.global.u64 [%3], %4; }"
                 :: "r"((unsigned)(on && blockIdx.x == 0)), "l"(g_finalize_phases + k), "l"(clk),
                    "l"(g_finalize_phases + kNumFinalizePhases + k), "l"(ns) : "memory");
}
extern "C" int irs_finalize_phases(unsigned long long* out) {
    return cudaMemcpyFromSymbol(out, g_finalize_phases, sizeof(g_finalize_phases)) == cudaSuccess ? 0 : 1;
}
#define IRS_FINALIZE_STAMP(k, cond) finalize_stamp(k, cond)
#else
#define IRS_FINALIZE_STAMP(k, cond) do { } while (0)
#endif

template <class Sys, int BT>
__global__ void __launch_bounds__(BT, 1) finalize_zero_order_kernel(const FinalizeArgs a) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    constexpr int NACC = gram_nacc(n, m);
    constexpr int WIDTH = gram_width_of<Sys>();      // NACC (+ first moments for centred-capable systems)
    __shared__ double Gm[d * d];      // Gram (then its Cholesky factor, lower)
    __shared__ double Bm[d * n];      // right-hand sides Z^T dF, then the solution
    __shared__ double sAB[n * d];
    __shared__ double inv_diag[d];
    __shared__ double nom[d + n];
    __shared__ double mom[WIDTH - NACC > 0 ? WIDTH - NACC : 1];   // [sum z' (d) | sum dF' (n)]
    __shared__ double spread[d];      // diagonal of the CENTRED Gram: scale of the rank test
    __shared__ double rho[n];         // centred: f_batch(2 xbar, 2 ubar) - f(xbar, ubar), the response shift
    __shared__ double colk[2][32];    // column k of the factor, for the lanes of warp 0
    const int tid = threadIdx.x, lane = tid & 31;
    const int p = blockIdx.x;
    IRS_FINALIZE_STAMP(kPhStart, tid == 0);
    // 0. sample-sharded run: exchange this point's chunk-reduced block with the other ranks first
    PartialSource src = partial_source(a);
    bool peer_late = false;
    int epoch = 0;
    if (a.peer.mode == kPeerExchange) epoch = peer_exchange_point<BT>(a, p, WIDTH, tid, &src, &peer_late);
    else if (a.peer.mode == kPeerGather) epoch = *reinterpret_cast<volatile int*>(a.peer.epoch) + 1;
    __shared__ int status_s;
    // 1. fixed-order sum over ranks and chunks, unpacked into the symmetric Gram and the rhs; a thread's
    //    entries over kFinalizeChunksInFlight chunks are summed together so that all their loads are in
    //    flight at once
    {
        constexpr int NE = (WIDTH + BT - 1) / BT;
        int rel[NE];
#pragma unroll
        for (int q = 0; q < NE; ++q) rel[q] = tid + q * BT < WIDTH ? tid + q * BT : -1;
        double sums[NE];
        const long long pbase = (long long)p * (src.reduced != nullptr ? (long long)WIDTH : (long long)src.C * WIDTH);
        sum_partials_multi<NE, kFinalizeChunksInFlight>(src, pbase, rel, WIDTH, sums);
        IRS_FINALIZE_STAMP(kPhSums, tid == 0);
#pragma unroll
        for (int q = 0; q < NE; ++q) {
            if (rel[q] >= NACC) {
                mom[rel[q] - NACC] = sums[q];
            } else if (rel[q] >= 0) {
                const int i = a.tables->gram_i[rel[q]], j = a.tables->gram_j[rel[q]];
                if (j < d) {
                    Gm[i * d + j] = sums[q];
                    Gm[j * d + i] = sums[q];
                } else {
                    Bm[i * n + (j - d)] = sums[q];
                }
            }
        }
    }
    if constexpr (WIDTH > NACC) {
        if (a.centered && tid == 32) {
            // response shift of the centred accumulation, in fp64 (the samples of a centred launch go
            // through the batch variant of the dynamics, the nominal response through the scalar one)
            const Sys sys(a.prm);
            double xb[n], ub[m], x2[n], u2[m], f2[n], fb[n];
#pragma unroll
            for (int q = 0; q < n; ++q) { xb[q] = a.x_nom[(long long)p * n + q];  x2[q] = 2.0 * xb[q]; }
#pragma unroll
            for (int q = 0; q < m; ++q) { ub[q] = a.u_nom[(long long)p * m + q];  u2[q] = 2.0 * ub[q]; }
            sys.template step<true>(x2, u2, f2);
            sys.template step<false>(xb, ub, fb);
#pragma unroll
            for (int q = 0; q < n; ++q) rho[q] = f2[q] - fb[q];
        }
    }
    __syncthreads();
    if (tid < d) spread[tid] = Gm[tid * d + tid];
    if constexpr (WIDTH > NACC) {
        // 1b. centred accumulation: z = s + z' with s = (xbar, ubar), dF = rho + dF', so
        //       Z^T Z  = Z'^T Z' + s m'^T + m' s^T + N s s^T
        //       Z^T dF = Z'^T dF' + m' rho^T + s g'^T + N s rho^T          (m' = sum z', g' = sum dF')
        //     in fp64.  The fp32 partials only ever held O(sigma) numbers.
        if (a.centered) {
            __syncthreads();      // spread[] read the centred diagonal
            for (int e = tid; e < d * d; e += BT) {
                const int i = e / d, j = e % d;
                const double si = i < n ? a.x_nom[(long long)p * n + i] : a.u_nom[(long long)p * m + (i - n)];
                const double sj = j < n ? a.x_nom[(long long)p * n + j] : a.u_nom[(long long)p * m + (j - n)];
                Gm[e] = fma(a.n_total * si, sj, fma(si, mom[j], fma(mom[i], sj, Gm[e])));
            }
            for (int e = tid; e < d * n; e += BT) {
                const int i = e / n, q = e % n;
                const double si = i < n ? a.x_nom[(long long)p * n + i] : a.u_nom[(long long)p * m + (i - n)];
                Bm[e] = fma(a.n_total * si, rho[q], fma(si, mom[d + q], fma(mom[i], rho[q], Bm[e])));
            }
        }
    }
    __syncthreads();
    IRS_FINALIZE_STAMP(kPhGram, tid == 0);
    // learned dynamics: warp 1 evaluates the network together (Mlp::step_warp, bit-identical to the functor)
    constexpr bool kWarpNominal = is_mlp<Sys>::value;
    __shared__ float mlp_act[kWarpNominal ? 2 * kMlpMaxHidden : 1];
    if (kWarpNominal ? (tid >= 32 && tid < 64) : (tid == 32)) {
        if constexpr (kWarpNominal) {
            const Sys sys(a.prm);
            double xb[n], ub[m], fb[n];
#pragma unroll
            for (int q = 0; q < n; ++q) xb[q] = a.x_nom[(long long)p * n + q];
#pragma unroll
            for (int q = 0; q < m; ++q) ub[q] = a.u_nom[(long long)p * m + q];
            sys.step_warp(xb, ub, fb, mlp_act, mlp_act + kMlpMaxHidden, tid - 32);
            if (tid == 32) {
#pragma unroll
                for (int q = 0; q < n; ++q) nom[q] = xb[q];
#pragma unroll
                for (int q = 0; q < m; ++q) nom[n + q] = ub[q];
#pragma unroll
                for (int q = 0; q < n; ++q) nom[n + m + q] = fb[q];
            }
        } else {
            nominal_compute_to_smem<Sys>(a, p, nom);
        }
        IRS_FINALIZE_STAMP(kPhNominal, tid == 32);
    } else if (tid < 32) {
        // 2. Cholesky G = L L^T by warp 0, right-looking, lane = row with the row of the factor in
        //    REGISTERS: once column k is scaled, its entries reach the other lanes (see below) and every
        //    lane updates its later entries with them; the pivot of column k + 1 is then one shuffle away
        //    and every lane computes its reciprocal square root (same operands: identical bits).  Each
        //    entry receives its updates in ascending column order — the fmas of the left-looking
        //    factorisation this replaces (and of the quad kernel), operand for operand — and only one
        //    update lies between two pivots, not two chains of k of them.
        //    A column whose diagonal is exactly zero (sigma = 0: regressor identically zero) gets
        //    coefficient 0, which is what the min-norm lstsq of the reference returns for it.
        bool bad = false;
        unsigned zero_mask = 0;
        double row[d];
#pragma unroll
        for (int j = 0; j < d; ++j) row[j] = (lane < d && j <= lane) ? Gm[lane * d + j] : 0.0;
        double piv = __shfl_sync(0xffffffffu, row[0], 0);      // G_kk - sum_{j<k} L_kj^2, updated by lane k
        static_for<0, d>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            const double d0 = Gm[k * d + k];      // the original diagonal entry G_kk (Gm is written after the loop)
            double dk = piv;
            // pivot <= 1e-6 * G_kk: the column is (numerically) a combination of earlier ones; the
            // fp32 partial sums carry ~1e-7 relative noise, so anything below is rank deficiency.
            // (Centred accumulation: the noise is relative to the SPREAD of the column, i.e. the centred
            //  diagonal, and a pivot of the shifted Gram is never below that of the centred one.)
            const double scale_k = (WIDTH > NACC && a.centered) ? spread[k] : d0;
            const bool zero_col = d0 == 0.0;
            const bool dependent = !zero_col && !(dk > 1e-6 * scale_k);
            bad = bad || dependent;
            if (zero_col || dependent) dk = 1.0;
            const double ikk = rsqrt(dk);           // one special function on the critical path, not two
            // selects, not branches: no reconvergence point between two pivots
            const double lik = zero_col ? 0.0 : row[k] * ikk, lkk = dk * ikk;
            row[k] = lane > k ? lik : (lane == k ? lkk : row[k]);
            if (lane == k) inv_diag[k] = ikk;
            if (zero_col) zero_mask |= 1u << k;
            // G_ic -= L_ik L_ck for every later column c.  The next pivot's column first, by shuffle, and
            // its pivot is broadcast at once; the other columns read L_ck from shared memory (one store
            // per lane instead of two shuffles per column; two buffers: a lane may store column k + 2
            // once every lane has passed the barrier of column k + 1, i.e. finished reading column k).
            if constexpr (k + 1 < d) {
                const double l = __shfl_sync(0xffffffffu, row[k], k + 1);      // L_k+1,k
                row[k + 1] = fma(-row[k], l, row[k + 1]);
                piv = __shfl_sync(0xffffffffu, row[k + 1], k + 1);
            }
            if constexpr (k + 2 < d) {
                double* col = colk[k & 1];
                col[lane] = row[k];
                __syncwarp();
                static_for<k + 2, d>([&](auto cc) {
                    constexpr int c = decltype(cc)::value;
                    row[c] = fma(-row[k], col[c], row[c]);      // col[c] = L_ck
                });
            }
        });
        for (int k = 0; k < d; ++k)
            if ((zero_mask >> k) & 1u)
                for (int q = lane; q < n; q += 32) Bm[k * n + q] = 0.0;
        if (lane < d) {
#pragma unroll
            for (int j = 0; j < d; ++j)
                if (j <= lane) Gm[lane * d + j] = row[j];      // the solves read the factor from shared memory
        }
        __syncwarp();
        IRS_FINALIZE_STAMP(kPhFactor, lane == 0);
        // 3. solve L L^T X = B, one right-hand side per lane (reciprocal diagonal: no divisions)
        if (lane < n) {
            const int q = lane;
            // fully unrolled, solution in registers, the L loads pipeline
            double y[d];
#pragma unroll
            for (int r = 0; r < d; ++r) {
                double s0 = Bm[r * n + q];
#pragma unroll
                for (int k = 0; k < r; ++k) s0 = fma(-Gm[r * d + k], y[k], s0);
                y[r] = s0 * inv_diag[r];
            }
#pragma unroll
            for (int r = d - 1; r >= 0; --r) {
                double s0 = y[r];
#pragma unroll
                for (int k = r + 1; k < d; ++k) s0 = fma(-Gm[k * d + r], y[k], s0);
                y[r] = s0 * inv_diag[r];
            }
#pragma unroll
            for (int r = 0; r < d; ++r) {
                if (!(y[r] == y[r]) || fabs(y[r]) > 1e300) bad = true;
                sAB[q * d + r] = y[r];      // [A|B] = X^T
            }
        }
        bad = __any_sync(0xffffffffu, bad);
        if (lane == 0) status_s = peer_late ? 2 : (bad ? 1 : 0);      // 2: a peer's block never arrived
        IRS_FINALIZE_STAMP(kPhSolve, lane == 0);
    }
    __syncthreads();
    if (a.peer.mode == kPeerGather) {
        write_abc_gather<Sys, BT>(a, p, sAB, nom, status_s, epoch, tid);
        peer_gather_finish<BT>(a, epoch, tid);
    } else {
        if (tid == 0) a.status[p] = status_s;
        write_abc<Sys, BT>(a, p, sAB, nom, tid);
        IRS_FINALIZE_STAMP(kPhWritten, tid == 0);
        if (a.peer.mode == kPeerExchange) peer_exchange_finish(a, epoch, tid);
    }
}

// ---------------------------------------------------------------------------------------------
// Finalize for many points (batched MPC: 4096 instances x T points): FOUR threads ("quad") per
// nominal point, 32 points per block.  The warp-per-point variant above spends a whole warp
// instruction on every scalar step of a 16 x 16 factorisation (136 useful lanes out of 16 x 5 x 32
// in the trailing update, 12 of 32 in the solves); here a warp carries eight points:
//   * the packed lower triangle of a point's Gram lives in shared memory as L[entry][point]
//     (1 KB per point, so a dozen warps per SM stay resident and hide the fp64 latencies);
//   * Cholesky, left-looking: for column k every quad thread recomputes the pivot (same operands,
//     same order: identical bits) and takes every fourth row below it; one __syncwarp per column;
//   * solves: each thread owns ceil(n / 4) right-hand sides, loaded straight from global memory
//     into registers and solved in place, L read from shared memory (quad-uniform broadcast);
// (Every multiply-add of the factorisation, the solves and c_t is an explicit fma() in both kernels:
// whether the compiler contracts a - b * c is its own choice, and one uncontracted update is one ulp.)
// The floating-point operations and their order are those of finalize_zero_order_kernel, entry by
// entry (left-looking here, right-looking there: each entry still receives its updates in ascending
// column order), so a point's result does not depend on which variant a launch picks — checked
// bit for bit by tests/test_gpu_parity.py::test_finalize_variants_are_bit_identical.
// ---------------------------------------------------------------------------------------------
constexpr int kFinalizeQuadThreads = 128;
constexpr int kQuad = 4;

template <class Sys>
struct FinalizeQuadCfg {
    static constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    static constexpr int W = d + n;
    static constexpr int NACC = gram_width_of<Sys>();      // stride of a packed partial block (the first
                                                           // moments of centred-capable systems are not read here)
    static constexpr int TRI = d * (d + 1) / 2;
    static constexpr int PPB = kFinalizeQuadThreads / kQuad;     // points per block
    static constexpr int QT = (n + kQuad - 1) / kQuad;           // right-hand sides per thread
    static constexpr int LDP = PPB + 1;                          // padded point stride (doubles)
    // Gram load slots: packed row i holds d - i Gram entries, ceil((d - i) / 4) per quad thread
    __host__ __device__ static constexpr int row_slots(int i) { return (d - i + kQuad - 1) / kQuad; }
    __host__ __device__ static constexpr int slot_offset(int i) {
        int o = 0;
        for (int r = 0; r < i; ++r) o += row_slots(r);
        return o;
    }
    static constexpr int GSLOTS = slot_offset(d);
    static constexpr size_t kSmemBytes = (size_t)(TRI + d) * LDP * sizeof(double);
};

template <class Sys>
__global__ void __launch_bounds__(kFinalizeQuadThreads, 3) finalize_zero_order_quad_kernel(const FinalizeArgs a) {
    using C = FinalizeQuadCfg<Sys>;
    constexpr int n = C::n, m = C::m, d = C::d, QT = C::QT, PPB = C::PPB, NACC = C::NACC;
    constexpr int LDP = C::LDP;
    extern __shared__ double fin_L[];            // [TRI][LDP]  packed lower triangle, (r, c) -> r (r + 1) / 2 + c
    double* fin_inv = fin_L + C::TRI * LDP;      // [d][LDP]    reciprocal pivots
    const int tid = threadIdx.x, g = tid & (kQuad - 1), pt = tid / kQuad;
    const long long p_raw = (long long)blockIdx.x * PPB + pt;
    const bool active = p_raw < a.P;
    // the quads past the last point redo the last point and write nothing (every lane then takes part
    // in the warp synchronisations and no lane factors garbage)
    const long long p = active ? p_raw : (long long)a.P - 1;
    // entries of one point inside a rank buffer: [C][width] fp32 partials or [width] fp64 reduced
    const long long pbase = p * (a.reduced != nullptr ? (long long)NACC : (long long)a.C * NACC);
#define IRS_L(r, c) fin_L[((r) * ((r) + 1) / 2 + (c)) * LDP + pt]

    // 1. Gram entries of the point -> shared memory: packed row i holds G[i][i..d-1] contiguously, the
    //    quad reads four consecutive entries at a time (fixed-order sum over ranks and chunks)
    {
        int rel[C::GSLOTS];
        static_for<0, d>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
#pragma unroll
            for (int t = 0; t < C::row_slots(i); ++t) {
                const int j = i + g + kQuad * t;
                rel[C::slot_offset(i) + t] = j < d ? gram_row_offset(i, C::W) + (j - i) : -1;
            }
        });
        double s[C::GSLOTS];
        sum_partials_multi<C::GSLOTS>(partial_source(a), pbase, rel, NACC, s);
        static_for<0, d>([&](auto ic) {
            constexpr int i = decltype(ic)::value;
#pragma unroll
            for (int t = 0; t < C::row_slots(i); ++t) {
                const int j = i + g + kQuad * t;
                if (j < d) fin_L[(j * (j + 1) / 2 + i) * LDP + pt] = s[C::slot_offset(i) + t];
            }
        });
    }
    __syncwarp();

    // 2. Cholesky G = L L^T.  A column whose diagonal is exactly zero (sigma = 0: regressor identically
    //    zero) gets coefficient 0, which is what the min-norm lstsq of the reference returns for it.
    bool bad = false;
    unsigned zero_mask = 0;
    static_for<0, d>([&](auto kc) {
        constexpr int k = decltype(kc)::value;
        double lk[k > 0 ? k : 1];            // row k of the factor (entries j < k)
        static_for<0, k>([&](auto jc) { constexpr int j = decltype(jc)::value;  lk[j] = IRS_L(k, j); });
        const double d0 = IRS_L(k, k);       // the original diagonal entry G_kk (never overwritten)
        double dk = d0;
        static_for<0, k>([&](auto jc) { constexpr int j = decltype(jc)::value;  dk = fma(-lk[j], lk[j], dk); });
        bool zero_col = false;
        // pivot <= 1e-6 * G_kk: the column is (numerically) a combination of earlier ones
        if (d0 == 0.0) { zero_col = true; dk = 1.0; }
        else if (!(dk > 1e-6 * d0)) { bad = true; dk = 1.0; }
        const double ikk = rsqrt(dk);
        if (g == 0) fin_inv[k * LDP + pt] = ikk;      // the solves only ever need the reciprocal pivot
#pragma unroll
        for (int t = 0; t < (d - 1 - k + kQuad - 1) / kQuad; ++t) {
            const int r = k + 1 + g + kQuad * t;
            if (r < d) {
                double* row = fin_L + (r * (r + 1) / 2) * LDP + pt;
                double s = row[k * LDP];
                static_for<0, k>([&](auto jc) { constexpr int j = decltype(jc)::value;  s = fma(-row[j * LDP], lk[j], s); });
                row[k * LDP] = zero_col ? 0.0 : s * ikk;
            }
        }
        if (zero_col) zero_mask |= 1u << k;
        __syncwarp();
    });

    // 3. right-hand sides of this thread (columns q = QT g .. QT g + QT - 1 of Z^T dF) -> registers,
    //    solved in place: L L^T X = B
    double y[d][QT];
    {
        constexpr int RH = (d + 1) / 2;          // two batches of rows: fewer loads (registers) in flight
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int rel[RH * QT];
#pragma unroll
            for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                for (int qq = 0; qq < QT; ++qq) {
                    const int r = h * RH + rr, q = QT * g + qq;
                    rel[rr * QT + qq] = (r < d && q < n && !((zero_mask >> r) & 1u))
                                            ? gram_row_offset(r, C::W) + (d - r) + q : -1;
                }
            double s[RH * QT];
            sum_partials_multi<RH * QT>(partial_source(a), pbase, rel, NACC, s);
#pragma unroll
            for (int rr = 0; rr < RH; ++rr)
#pragma unroll
                for (int qq = 0; qq < QT; ++qq)
                    if (h * RH + rr < d) y[h * RH + rr][qq] = s[rr * QT + qq];
        }
    }
    static_for<0, d>([&](auto rc) {
        constexpr int r = decltype(rc)::value;
        static_for<0, r>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            const double l = IRS_L(r, k);
#pragma unroll
            for (int qq = 0; qq < QT; ++qq) y[r][qq] = fma(-l, y[k][qq], y[r][qq]);
        });
        const double inv = fin_inv[r * LDP + pt];
#pragma unroll
        for (int qq = 0; qq < QT; ++qq) y[r][qq] *= inv;
    });
    // (compiler fence: without it the factor entries loaded by the forward pass are kept for the
    //  backward pass — 136 doubles — and spill)
    __syncwarp();
    static_for<0, d>([&](auto rc) {
        constexpr int r = d - 1 - decltype(rc)::value;
        static_for<r + 1, d>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            const double l = IRS_L(k, r);
#pragma unroll
            for (int qq = 0; qq < QT; ++qq) y[r][qq] = fma(-l, y[k][qq], y[r][qq]);
        });
        const double inv = fin_inv[r * LDP + pt];
#pragma unroll
        for (int qq = 0; qq < QT; ++qq) y[r][qq] *= inv;
    });
    // 4. [A|B] = X^T and c = f(xbar, ubar) - A xbar - B ubar (f(xbar, ubar) was written to ct)
#pragma unroll
    for (int qq = 0; qq < QT; ++qq) {
        const int q = QT * g + qq;
        if (q < n) {
            double acc = a.ct[p * n + q];
#pragma unroll
            for (int r = 0; r < d; ++r) {
                const double v = y[r][qq];
                if (!(v == v) || fabs(v) > 1e300) bad = true;
                if (active) {
                    if (r < n) a.At[(p * n + q) * n + r] = v;
                    else a.Bt[(p * n + q) * m + (r - n)] = v;
                }
                acc = fma(-v, r < n ? a.x_nom[p * n + r] : a.u_nom[p * m + (r - n)], acc);
            }
            if (active) a.ct[p * n + q] = acc;
        }
    }
    // a point is flagged if any of its quad threads saw a bad pivot or a non-finite coefficient
    bad = __any_sync(0xfu << (4 * ((tid & 31) / 4)), bad);
    if (active && g == 0) a.status[p] = bad ? 1 : 0;
#undef IRS_L
}

template <class Sys>
__global__ void __launch_bounds__(kFinalizeThreads) finalize_first_order_kernel(const FinalizeArgs a) {
    constexpr int n = Sys::N, d = Sys::D;
    constexpr int NJ = Sys::NJ > 0 ? Sys::NJ : 1;
    __shared__ double sV[NJ];
    __shared__ double sAB[n * d];
    __shared__ double nom[d + n];
    const int tid = threadIdx.x;
    const int p = blockIdx.x;
    const Sys sys(a.prm);
    PartialSource src = partial_source(a);
    bool peer_late = false;
    int epoch = 0;
    if (a.peer.mode == kPeerExchange) epoch = peer_exchange_point<kFinalizeThreads>(a, p, NJ, tid, &src, &peer_late);
    else if (a.peer.mode == kPeerGather) epoch = *reinterpret_cast<volatile int*>(a.peer.epoch) + 1;
    for (int e = tid; e < NJ; e += kFinalizeThreads) sV[e] = sum_partials(src, p, e, NJ) / a.n_total;
    nominal_to_smem<Sys, kFinalizeThreads>(a, p, nom, tid);
    __syncthreads();
    if (tid == 0) {
        double v[NJ], J[n * d];
        for (int k = 0; k < NJ; ++k) v[k] = sV[k];
        sys.jac_assemble(v, J);
        for (int e = 0; e < n * d; ++e) sAB[e] = J[e];
        if (a.peer.mode != kPeerGather) a.status[p] = peer_late ? 2 : 0;
    }
    __syncthreads();
    if (a.peer.mode == kPeerGather) {
        write_abc_gather<Sys, kFinalizeThreads>(a, p, sAB, nom, 0, epoch, tid);
        peer_gather_finish<kFinalizeThreads>(a, epoch, tid);
    } else {
        write_abc<Sys, kFinalizeThreads>(a, p, sAB, nom, tid);
        if (a.peer.mode == kPeerExchange) peer_exchange_finish(a, epoch, tid);
    }
}

// Chunk reduction [P, C, width] fp32 -> [P, width] fp64 in fixed chunk order: the block a rank
// contributes to the sample-sharded exchange (all-gather of per-point Gram blocks).
__global__ void __launch_bounds__(256) reduce_chunks_kernel(const float* partials, int P, int C,
                                                           int width, double* reduced) {
    const long long total = (long long)P * width;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const long long p = idx / width;
        const int e = (int)(idx % width);
        reduced[idx] = sum_chunks_in_order(partials + (p * C) * width + e, C, width);
    }
}

// ---------------------------------------------------------------------------------------------
// Exact linearization at the nominal points, all in fp64 (irs_lqr_exact.py:15-31):
// [A|B] = jacobian_xu(xbar, ubar), c = f(xbar, ubar) - A xbar - B ubar.  One thread per point.
// ---------------------------------------------------------------------------------------------
template <class Sys>
__global__ void __launch_bounds__(64) exact_linearize_kernel(SysParams prm, const double* x_nom,
                                                            const double* u_nom, int P, double* At,
                                                            double* Bt, double* ct) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    constexpr int NJ = Sys::NJ > 0 ? Sys::NJ : 1;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const Sys sys(prm);
    double xb[n], ub[m], fb[n], v[NJ], J[n * d];
#pragma unroll
    for (int q = 0; q < n; ++q) xb[q] = x_nom[(long long)p * n + q];
#pragma unroll
    for (int q = 0; q < m; ++q) ub[q] = u_nom[(long long)p * m + q];
    sys.jac_var(xb, ub, v);
    sys.jac_assemble(v, J);
    sys.template step<false>(xb, ub, fb);
#pragma unroll
    for (int r = 0; r < n; ++r) {
        double acc = fb[r];
#pragma unroll
        for (int q = 0; q < n; ++q) {
            At[((long long)p * n + r) * n + q] = J[r * d + q];
            acc -= J[r * d + q] * xb[q];
        }
#pragma unroll
        for (int q = 0; q < m; ++q) {
            Bt[((long long)p * n + r) * m + q] = J[r * d + n + q];
            acc -= J[r * d + n + q] * ub[q];
        }
        ct[(long long)p * n + r] = acc;
    }
}

// ---------------------------------------------------------------------------------------------
// Debug / bookkeeping kernel: dump the Philox words and the deltas exactly as the fused kernels
// draw them (same counter function).  Used by the bit-exact index tests.
// ---------------------------------------------------------------------------------------------
struct PhiloxDumpArgs {
    int P, d;
    long long N;
    uint32_t seed_lo, seed_hi, iter, stream, p0;
    unsigned long long i0;
    int antithetic;          // samples 2q, 2q + 1 = +z_q, -z_q (one counter per pair)
    uint32_t* words;
    float* deltas;
    float sigma_scaled[16];
};

__global__ void philox_dump_kernel(const PhiloxDumpArgs a) {
    const int nblk = (a.d + 3) / 4;
    const long long total = (long long)a.P * a.N * nblk;
    for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
         idx += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(idx % nblk);
        const long long i = (idx / nblk) % a.N;
        const int p = (int)(idx / nblk / a.N);
        uint32_t r[4];
        unsigned long long gi = a.i0 + (unsigned long long)i;
        float sg = 1.f;
        if (a.antithetic) {
            sg = (gi & 1ull) ? -1.f : 1.f;
            gi >>= 1;
        }
        philox4x32((uint32_t)gi, a.p0 + (uint32_t)p, (a.iter << 8) | (uint32_t)j, a.stream, a.seed_lo, a.seed_hi, r);
        if (a.words != nullptr)
            for (int q = 0; q < 4; ++q) a.words[idx * 4 + q] = r[q];
        if (a.deltas != nullptr) {
            float e[4];
            box_muller_raw(r[0], r[1], e[0], e[1]);
            box_muller_raw(r[2], r[3], e[2], e[3]);
            for (int q = 0; q < 4; ++q)
                if (4 * j + q < a.d)
                    a.deltas[((long long)p * a.N + i) * a.d + 4 * j + q] = sg * (a.sigma_scaled[4 * j + q] * e[q]);
        }
    }
}

}  // namespace irs
