// extern "C" entry points declared in include/irs_mpc_b200.h: argument validation + launches.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "../../include/irs_mpc_b200.h"
#include "smooth.cuh"
#include "smooth_tc.cuh"
#include "tvlqr.cuh"
#include "tvlqr_box.cuh"
#include "tvlqr_any.cuh"
#include "cem.cuh"
#include "smooth_mlp.cuh"

namespace irs {

static thread_local char g_error[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
}

int check_launch(const char* what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

// Registered networks of the learned-dynamics system (irs_mlp_register): device blobs, one per handle.
struct MlpEntry {
    float* blob;
    unsigned short* w2_tc;      // [W2 | b2] as K-major bf16 operand pieces (smooth_mlp.cuh: MlpTcLayout)
    int d, n, h1, h2, device;
};
static std::vector<MlpEntry> g_mlps;
static std::mutex g_mlp_mutex;

static int load_params(int system, const double* params_host, int nparams, SysParams* out) {
#ifndef IRS_USER_SYSTEM
    static const int expected[kNumSystems] = {1, 1, 9, 2, 2};
#else
    static const int expected[kNumSystems] = {1, 1, 9, 2, 2, IRS_USER_NPARAMS};
#endif
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    IRS_REQUIRE(params_host != nullptr && nparams == expected[system],
                "system %d expects %d parameters, got %d", system, expected[system], nparams);
    memset(out, 0, sizeof(*out));
    for (int i = 0; i < nparams; ++i) {
        out->v[i] = params_host[i];
        out->f[i] = (float)params_host[i];
    }
    if (system == kMlp21) {          // [h, handle] -> the registered network
        const int handle = (int)params_host[1];
        std::lock_guard<std::mutex> lock(g_mlp_mutex);
        IRS_REQUIRE(handle >= 0 && handle < (int)g_mlps.size() && g_mlps[handle].blob != nullptr,
                    "unknown network handle %d (irs_mlp_register)", handle);
        const MlpEntry& e = g_mlps[handle];
        const SystemDims dm = system_dims(system);
        IRS_REQUIRE(e.n == dm.n && e.d == dm.n + dm.m, "network %d maps %d -> %d, system %d needs %d -> %d", handle,
                    e.d, e.n, system, dm.n + dm.m, dm.n);
        int dev = 0;
        cudaGetDevice(&dev);
        IRS_REQUIRE(dev == e.device, "network %d was registered on device %d, current device is %d", handle, e.device, dev);
        out->mlp = e.blob;
        out->mlp_w2 = e.w2_tc;
        out->h1 = e.h1;
        out->h2 = e.h2;
    }
    if (system == kQuadrotor) {      // derived invariants of Quadrotor<float>::step, rounded once
        const double* v = out->v;    // [h, mass, L, g, Ixx, Iyy, Izz, kF, kM]
        out->f[9] = (float)(1.0 / v[1]);
        out->f[10] = (float)(1.0 / v[4]);
        out->f[11] = (float)(1.0 / v[5]);
        out->f[12] = (float)(1.0 / v[6]);
        out->f[13] = (float)(v[2] * v[7]);
        out->f[14] = (float)(v[5] - v[6]);
        out->f[15] = (float)(v[6] - v[4]);
        out->f[16] = (float)(v[4] - v[5]);
    }
    return 0;
}

// The accumulate kernel launched last on this thread: irs_graph_end looks its node up in a captured
// graph so that irs_graph_update_smoothing can re-parameterise it (seed, iter, sigma) per replay.
static thread_local const void* g_last_smooth_func = nullptr;

template <class Sys, int G>
static int launch_zero_order(const SmoothArgs& a, cudaStream_t st) {
    using C = ZeroOrderCfg<Sys, G>;
    const size_t smem = G == 1 ? sizeof(float) * (C::kThreads / 32) * gram_width_of<Sys>()
                               : sizeof(float) * 2 * C::kTile * C::RS;      // double-buffered tile
    auto kern = smooth_zero_order_kernel<Sys, G>;
    if (smem > 48 * 1024) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(smooth_zero_order)");
    }
    g_last_smooth_func = (const void*)kern;
    kern<<<(unsigned)((long long)a.P * a.C), C::kThreads, smem, st>>>(a);
    return check_launch("smooth_zero_order_kernel");
}

// Gram engine of the zero-order kernel: -1 = auto (tensor cores when the regressor dimension is
// large enough to pay for the operand staging: quadrotor, three_cart), 0 = CUDA cores (FFMA2), 1 = tcgen05.
static int g_gram_engine = -2;
static int gram_engine() {
    if (g_gram_engine == -2) {
        const char* e = getenv("IRS_GRAM_ENGINE");
        g_gram_engine = e ? atoi(e) : -1;
        if (g_gram_engine < -1 || g_gram_engine > 1) g_gram_engine = -1;
    }
    return g_gram_engine;
}
static bool use_tensor_cores(int system) {
    const int e = gram_engine();
#ifdef IRS_USER_SYSTEM
    // user system: CUDA cores up to 8 regressors (as for pendulum and bicycle), tcgen05 above
    if (e == -1) return system == kUser && UserSystem<float>::D > 8;
#endif
    if (e == -1) return system == kQuadrotor || system == kThreeCart;   // measured: see DESIGN.md
    return e == 1;
}
static int num_sms() {
    static int cached[64] = {0};      // per device (one process may drive several GPUs)
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// Learned dynamics: hidden layer on the tensor cores (smooth_mlp.cuh).  Persistent grid of the blocks that are
// resident together; IRS_MLP_ENGINE=0 selects the generic per-thread functor instead (parity tests).
template <class Sys>
static int launch_zero_order_mlp(const SmoothArgs& a, cudaStream_t st) {
    const MlpTcLayout L(a.prm.h1, a.prm.h2);
    auto kern = smooth_zero_order_mlp_kernel<Sys>;
    static int max_smem = 0, per_sm_smem = 0;
    if (max_smem == 0) {
        int dev = 0, optin = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cudaDeviceGetAttribute(&per_sm_smem, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(smooth_zero_order_mlp)");
        max_smem = optin;
    }
    // Tile groups per block and blocks per SM (1 KB of shared memory reserved per block, 512 TMEM columns per SM).
    // Two one-group blocks per SM were measured faster than one block of two or three groups (the reference's
    // 100 / 100 network: 0.272 against 0.305 / 0.289 ms); wider networks, whose operand tiles leave room for one
    // block only, take as many groups as fit.
    const int max_groups = MlpTcSmem<Sys>::groups_for(L, max_smem);
    IRS_REQUIRE(max_groups >= 1, "hidden widths %d / %d need %d bytes of shared memory (limit %d)", L.H1, L.H2,
                MlpTcSmem<Sys>(L, 1).total, max_smem);
    const int groups = per_sm_smem / (MlpTcSmem<Sys>(L, 1).total + 1024) >= 2 ? 1 : max_groups;
    const MlpTcSmem<Sys> sm(L, groups);
    int per_sm = per_sm_smem / (sm.total + 1024);
    const int tmem_cols = MlpTcLayout::tmem_alloc_cols(groups * L.tmem_cols_per_group());
    if (per_sm > 512 / tmem_cols) per_sm = 512 / tmem_cols;
    if (per_sm < 1) per_sm = 1;
    const long long items = (long long)a.P * a.C;
    const long long resident = (long long)per_sm * num_sms();
    const long long want = (items + groups - 1) / groups;       // every group is a worker with its own items
    g_last_smooth_func = (const void*)kern;
    kern<<<(unsigned)(want < resident ? want : resident), 128 * groups, (size_t)sm.total, st>>>(a);
    return check_launch("smooth_zero_order_mlp_kernel");
}
static bool use_mlp_tensor_cores() {
    const char* e = getenv("IRS_MLP_ENGINE");      // read per call: the parity tests switch engines
    return !(e != nullptr && atoi(e) == 0);
}

template <class Sys, int MODE, bool CENTERED>
static int launch_zero_order_tc_mode(const SmoothArgs& a, cudaStream_t st) {
    using C = TcCfg<Sys, MODE == kTcPaired && Sys::kHasProjection>;
    constexpr int NSTAGE = 1;      // measured: one tile per warp is fastest (DESIGN.md)
    const size_t smem = (size_t)NSTAGE * C::kWarps * C::kStageBytes;
    auto kern = smooth_zero_order_tc_kernel<Sys, NSTAGE, MODE, CENTERED>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(smooth_zero_order_tc)");
        // resident blocks per SM from the kernel's own resource usage (the occupancy API answers for
        // the *current* shared-memory carve-out, which is not the one the launch will configure)
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) return check_launch("cudaFuncGetAttributes");
        const int regs_per_block = ((fa.numRegs * 32 + 255) / 256 * 256) * (C::kThreads / 32);
        const int by_regs = 65536 / regs_per_block;
        const int by_smem = (int)((227 * 1024) / (smem + fa.sharedSizeBytes + 1024));
        const int by_tmem = 512 / C::kTmemCols;
        int occ = by_regs < by_smem ? by_regs : by_smem;
        if (by_tmem < occ) occ = by_tmem;
        if (occ > 32) occ = 32;
        blocks_per_sm = occ < 1 ? 1 : occ;
    }
    // persistent grid: every resident block walks the (point, chunk) item list with stride gridDim.x
    const long long items = (long long)a.P * a.C;
    long long grid = (long long)num_sms() * blocks_per_sm;
    if (grid > items) grid = items;
    g_last_smooth_func = (const void*)kern;
    kern<<<(unsigned)grid, C::kThreads, smem, st>>>(a);
    return check_launch("smooth_zero_order_tc_kernel");
}

template <class Sys, bool CENTERED>
static int launch_zero_order_tc_centered(const SmoothArgs& a, cudaStream_t st) {
    // the noise source is a compile-time mode of the kernel: replayed deltas, the Philox stream with one
    // draw per sample, or the Philox stream in antithetic pairs (one draw and one operand row per pair)
    if (a.noise != nullptr) return launch_zero_order_tc_mode<Sys, kTcReplay, CENTERED>(a, st);
    if (a.flags & kFlagAntithetic) return launch_zero_order_tc_mode<Sys, kTcPaired, CENTERED>(a, st);
    return launch_zero_order_tc_mode<Sys, kTcPhilox, CENTERED>(a, st);
}

template <class Sys>
static int launch_zero_order_tc(const SmoothArgs& a, cudaStream_t st) {
    if constexpr (Sys::kHasProjection) {      // centred-capable: absolute regressors accumulate relative to the nominal
        if (a.flags & (kFlagProjectAbsolute | kFlagCentered)) return launch_zero_order_tc_centered<Sys, true>(a, st);
    }
    return launch_zero_order_tc_centered<Sys, false>(a, st);
}

#ifdef IRS_USER_SYSTEM
// CUDA-core Gram engine of the user system: the whole block in every thread's registers up to 8 regressors;
// above that its rows are split over the four warps of a block (the quadrotor's layout), which needs a split
// that gives every warp the same number of outputs.
static int launch_zero_order_user(const SmoothArgs& a, cudaStream_t st) {
    using Sys = UserSystem<float>;
    if constexpr (Sys::D <= 8) {
        return launch_zero_order<Sys, 1>(a, st);
    } else {
        using C = ZeroOrderCfg<Sys, 4>;
        constexpr int NP = role_pairs(C::d, C::Wp, 4, 0);
        if constexpr (role_pairs(C::d, C::Wp, 4, 1) == NP && role_pairs(C::d, C::Wp, 4, 2) == NP &&
                      role_pairs(C::d, C::Wp, 4, 3) == NP) {
            IRS_REQUIRE(a.S % 128 == 0, "chunk size must be a multiple of 128");
            return launch_zero_order<Sys, 4>(a, st);
        } else {
            set_error("the CUDA-core Gram engine cannot split the rows of d = %d regressors evenly over four warps: "
                      "use the tensor-core engine (irs_set_gram_engine(-1) or (1))", Sys::D);
            return 1;
        }
    }
}
#endif

static int fill_smooth_args(SmoothArgs* a, int system, const double* params_host, int nparams,
                            int flags, const double* x_nom, const double* u_nom, int P, long long N,
                            const float* sigma, const float* noise, unsigned long long seed,
                            unsigned iter, unsigned stream_id, unsigned p0, unsigned long long i0,
                            int C, long long S, float* partials) {
    if (load_params(system, params_host, nparams, &a->prm)) return 1;
    IRS_REQUIRE(x_nom && u_nom && partials, "null pointer argument");
    IRS_REQUIRE(P >= 1 && N >= 1, "need at least one nominal point and one sample (P=%d, N=%lld)", P, N);
    IRS_REQUIRE(C >= 1 && S >= 1 && (long long)C * S >= N, "chunk plan (C=%d, S=%lld) does not cover N=%lld", C, S, N);
    IRS_REQUIRE((long long)P * C < (1ll << 31), "grid too large");
    IRS_REQUIRE(noise != nullptr || sigma != nullptr, "need either replayed noise or sigma");
    {
        const SystemDims dm = system_dims(system);
        a->nreg = dm.n + dm.m;
        for (int c = 0; c < kMaxRegressors; ++c)
            a->sigma_scaled[c] = (sigma != nullptr && c < dm.n + dm.m) ? kBoxMullerScale * sigma[c] : 0.f;
    }
    IRS_REQUIRE(iter < (1u << 24), "iter out of range");
    IRS_REQUIRE(!((flags & (IRS_PROJECT_ABSOLUTE | IRS_PROJECT_DELTA)) && system != kThreeCart),
                "projection flags are only defined for three_cart");
    IRS_REQUIRE(!((flags & IRS_PROJECT_ABSOLUTE) && (flags & IRS_PROJECT_DELTA)),
                "IRS_PROJECT_ABSOLUTE and IRS_PROJECT_DELTA are exclusive");
    IRS_REQUIRE(!((flags & IRS_ANTITHETIC) && noise == nullptr && (i0 & 1ull)),
                "antithetic pairs: the global index of the first local sample (i0) must be even");
    if (noise != nullptr) flags &= ~IRS_ANTITHETIC;      // replayed deltas are whatever the caller drew
    IRS_REQUIRE(!(flags & IRS_CENTERED) || system == kThreeCart,
                "centred accumulation (IRS_CENTERED) is built for three_cart only");
    IRS_REQUIRE(!(flags & IRS_CENTERED) || !(flags & IRS_PROJECT_DELTA), "IRS_CENTERED and IRS_PROJECT_DELTA are exclusive");
    a->x_nom = x_nom;  a->u_nom = u_nom;  a->noise = noise;
    a->partials = partials;  a->N = N;  a->S = S;  a->P = P;  a->C = C;
    a->seed_lo = (uint32_t)(seed & 0xffffffffull);
    a->seed_hi = (uint32_t)(seed >> 32);
    a->iter = iter;  a->stream = stream_id;  a->p0 = p0;  a->i0 = i0;  a->flags = flags;
    return 0;
}

template <typename R, class Sys>
__global__ void __launch_bounds__(128) dyn_batch_kernel(SysParams prm, int batch_variant, const R* x,
                                                        const R* u, R* out, long long B) {
    constexpr int n = Sys::N, m = Sys::M;
    const Sys sys(prm);
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        R xs[n], us[m], o[n];
#pragma unroll
        for (int q = 0; q < n; ++q) xs[q] = x[b * n + q];
#pragma unroll
        for (int q = 0; q < m; ++q) us[q] = u[b * m + q];
        if (batch_variant) sys.template step<true>(xs, us, o);
        else sys.template step<false>(xs, us, o);
#pragma unroll
        for (int q = 0; q < n; ++q) out[b * n + q] = o[q];
    }
}

template <typename R, class Sys>
__global__ void __launch_bounds__(128) jac_batch_kernel(SysParams prm, const R* x, const R* u, R* J,
                                                        long long B) {
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    constexpr int NJ = Sys::NJ > 0 ? Sys::NJ : 1;
    const Sys sys(prm);
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        R xs[n], us[m], v[NJ], Jl[n * d];
#pragma unroll
        for (int q = 0; q < n; ++q) xs[q] = x[b * n + q];
#pragma unroll
        for (int q = 0; q < m; ++q) us[q] = u[b * m + q];
        sys.jac_var(xs, us, v);
        sys.jac_assemble(v, Jl);
#pragma unroll
        for (int q = 0; q < n * d; ++q) J[b * n * d + q] = Jl[q];
    }
}

template <typename R, class Sys>
__global__ void __launch_bounds__(128) project_batch_kernel(SysParams prm, R* x, long long B) {
    constexpr int n = Sys::N;
    const Sys sys(prm);
    for (long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x; b < B;
         b += (long long)gridDim.x * blockDim.x) {
        R xs[n];
#pragma unroll
        for (int q = 0; q < n; ++q) xs[q] = x[b * n + q];
        sys.project(xs);
#pragma unroll
        for (int q = 0; q < n; ++q) x[b * n + q] = xs[q];
    }
}

// FP32 FMA peak microbenchmark (roofline denominator measured on the box): 8 independent
// dependent-FMA chains per thread, 148*8 blocks of 256 threads.
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters, float b, float c) {
    float acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = (float)(threadIdx.x + k);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = fmaf(acc[k], b, c);
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += acc[k];
    out[blockIdx.x * (long long)blockDim.x + threadIdx.x] = s;
}

static unsigned grid_for(long long work, int threads) {
    long long g = (work + threads - 1) / threads;
    if (g < 1) g = 1;
    if (g > 148 * 32) g = 148 * 32;
    return (unsigned)g;
}

template <typename R>
static int dynamics_batch_impl(int system, const double* params_host, int nparams, int batch_variant,
                               const R* x, const R* u, R* out, long long B, void* stream) {
    SysParams prm;
    if (load_params(system, params_host, nparams, &prm)) return 1;
    IRS_REQUIRE(B >= 0, "negative batch");
    if (B == 0) return 0;
    IRS_REQUIRE(x && u && out, "null pointer argument");
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_SYSTEM(system, R, Sys,
                        (dyn_batch_kernel<R, Sys><<<grid_for(B, 128), 128, 0, st>>>(prm, batch_variant, x, u, out, B)));
    return check_launch("dynamics_batch_kernel");
}

template <typename R>
static int jacobian_batch_impl(int system, const double* params_host, int nparams, const R* x,
                               const R* u, R* J, long long B, void* stream) {
    SysParams prm;
    if (load_params(system, params_host, nparams, &prm)) return 1;
    IRS_REQUIRE(system != kThreeCart,
                "three_cart is not differentiable and has no Jacobian (three_cart_dynamics.py:20)");
#ifdef IRS_USER_SYSTEM
    IRS_REQUIRE(UserSystem<double>::kHasJacobian, "the user system was built without a Jacobian body");
#endif
    IRS_REQUIRE(B >= 0, "negative batch");
    if (B == 0) return 0;
    IRS_REQUIRE(x && u && J, "null pointer argument");
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_SYSTEM(system, R, Sys,
                        (jac_batch_kernel<R, Sys><<<grid_for(B, 128), 128, 0, st>>>(prm, x, u, J, B)));
    return check_launch("jacobian_batch_kernel");
}

#ifndef IRS_USER_SYSTEM
#define IRS_DISPATCH_DIMS(n, m, ...)                                                \
    if (n == 2 && m == 1) { constexpr int N_ = 2, M_ = 1; __VA_ARGS__; }            \
    else if (n == 5 && m == 2) { constexpr int N_ = 5, M_ = 2; __VA_ARGS__; }       \
    else if (n == 12 && m == 4) { constexpr int N_ = 12, M_ = 4; __VA_ARGS__; }     \
    else if (n == 6 && m == 2) { constexpr int N_ = 6, M_ = 2; __VA_ARGS__; }       \
    else { irs::set_error("unsupported TVLQR dims n=%d m=%d", n, m); return 1; }
#else
// A user library holds the compile-time LQR kernels of its own system's pair only.  The Riccati pass and the
// linear rollout of a pair that is not a built-in one take the run-time-dimension kernels (tvlqr_any.cuh):
// the templated Riccati kernel's Cholesky is built for m in {1, 2, 4}, the tiled and packed kernels for fixed
// shapes.
#define IRS_DISPATCH_DIMS(n, m, ...)                                                                     \
    if (n == IRS_USER_N && m == IRS_USER_M) { constexpr int N_ = IRS_USER_N, M_ = IRS_USER_M; __VA_ARGS__; } \
    else { irs::set_error("unsupported TVLQR dims n=%d m=%d (this library is built for n=%d m=%d)", n, m,  \
                          IRS_USER_N, IRS_USER_M); return 1; }
#define IRS_USER_BUILTIN_DIMS                                                                             \
    ((IRS_USER_N == 2 && IRS_USER_M == 1) || (IRS_USER_N == 5 && IRS_USER_M == 2) ||                      \
     (IRS_USER_N == 12 && IRS_USER_M == 4) || (IRS_USER_N == 6 && IRS_USER_M == 2))
#endif

}  // namespace irs

using namespace irs;

// Rollout launch: systems whose next angles do not depend on the input take the two-warp kernel that
// evaluates the trigonometry one step ahead (IRS_ROLLOUT_TRIG=0 keeps the one-warp kernel; both give
// the same bits).
template <class Sys, bool CLOSED>
static void launch_rollout(const RolloutArgs& a, cudaStream_t st) {
    if constexpr (Sys::kTrigAhead > 0) {
        // few instances only: with thousands of instances the second warp per instance costs more
        // than the shorter critical path gains (4096 quadrotors: 0.66 ms against 0.45 ms)
        const char* e = getenv("IRS_ROLLOUT_TRIG");
        if (e != nullptr ? atoi(e) != 0 : a.I <= 2 * num_sms()) {
            rollout_trig_kernel<Sys, CLOSED><<<(unsigned)a.I, 64, 0, st>>>(a);
            return;
        }
    }
    if constexpr (is_mlp<Sys>::value) {
        // learned dynamics: one block per instance with the network in registers
        rollout_mlp_kernel<Sys, CLOSED><<<(unsigned)a.I, kMlpMaxHidden, 0, st>>>(a);
    } else {
        rollout_kernel<Sys, CLOSED><<<(a.I + kRolloutWarps - 1) / kRolloutWarps, 32 * kRolloutWarps, 0, st>>>(a);
    }
}

template <class Sys>
static int launch_box_mpc(const BoxMpcArgs& a, cudaStream_t st) {
    // stage the per-step matrices in shared memory when they fit next to the ADMM state
    const size_t with_cache = box_mpc_smem_bytes<Sys::N, Sys::M>(a.T, true);
    const bool cache = with_cache <= 200 * 1024;
    const size_t smem = cache ? with_cache : box_mpc_smem_bytes<Sys::N, Sys::M>(a.T, false);
    IRS_REQUIRE(smem <= 200 * 1024, "horizon T=%d too long for the shared-memory resident ADMM state", a.T);
    if (cache) {
        auto kern = box_mpc_kernel<Sys, true>;
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(box_mpc_kernel)");
        kern<<<(unsigned)a.I, 32, smem, st>>>(a);
    } else {
        auto kern = box_mpc_kernel<Sys, false>;
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(box_mpc_kernel)");
        kern<<<(unsigned)a.I, 32, smem, st>>>(a);
    }
    return check_launch("box_mpc_kernel");
}

extern "C" {

int irs_abi_version(void) { return IRS_ABI_VERSION; }

const char* irs_last_error(void) { return g_error; }

int irs_set_gram_engine(int engine) {
    IRS_REQUIRE(engine >= -1 && engine <= 1, "engine must be -1 (auto), 0 (CUDA cores) or 1 (tensor cores)");
    g_gram_engine = engine;
    return 0;
}

int irs_system_dims(int system, int* n, int* m, int* nj) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    const SystemDims d = system_dims(system);
    if (n) *n = d.n;
    if (m) *m = d.m;
    if (nj) *nj = d.nj;
    return 0;
}

int irs_partial_width(int system, int order) {
    if (system < 0 || system >= kNumSystems) return -1;
    const SystemDims d = system_dims(system);
    // three_cart blocks carry the first moments of the centred accumulation (smooth.cuh: gram_width)
    return order == 0 ? gram_width(d.n, d.m, system == kThreeCart) : (d.nj > 0 ? d.nj : 1);
}

int irs_smooth_plan(int system, int order, int P, long long N, long long chunk_samples, int* C, long long* S) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    IRS_REQUIRE(P >= 1 && N >= 1 && C && S && chunk_samples >= 0, "bad plan arguments");
    // Samples per chunk: large enough to amortise the end-of-chunk reduction, small enough that
    // P*C blocks give several waves over 148 SMs.  The plan depends on N (and on the caller's
    // chunk_samples) ONLY, never on P, so that a timestep-sharded run (P split over ranks) sums in
    // exactly the same order as the single-GPU run and reproduces it bit for bit.
    // chunk_samples = 0: the default target of 4096; callers whose launches are smaller than a resident
    // grid (strong scaling) ask for smaller chunks so that every SM still holds several work items.
    const long long tile = 256;        // a block round: 128 lanes x (one sample | one antithetic pair)
    long long target = 4096;
    if (system == kMlp21 && order == 0) target = 1536;   // 12 tiles of 128 for up to 3 tile groups; several waves of items
    if (chunk_samples > 0) target = chunk_samples;
    long long c = (N + target - 1) / target;
    long long s = (N + c - 1) / c;
    s = (s + tile - 1) / tile * tile;
    c = (N + s - 1) / s;
    *C = (int)c;
    *S = s;
    return 0;
}

int irs_smooth_zero_order_accumulate(int system, const double* params_host, int nparams, int flags,
                                     const double* x_nom, const double* u_nom, int P, long long N,
                                     const float* sigma_host, const float* noise,
                                     unsigned long long seed, unsigned iter, unsigned stream_id,
                                     unsigned p0, unsigned long long i0,
                                     int C, long long S, float* partials, void* stream) {
    SmoothArgs a;
    if (fill_smooth_args(&a, system, params_host, nparams, flags, x_nom, u_nom, P, N, sigma_host, noise,
                         seed, iter, stream_id, p0, i0, C, S, partials))
        return 1;
    cudaStream_t st = (cudaStream_t)stream;
    if (use_tensor_cores(system)) {
        switch (system) {
#ifndef IRS_USER_SYSTEM
            case kPendulum: return launch_zero_order_tc<Pendulum<float>>(a, st);
            case kBicycle: return launch_zero_order_tc<Bicycle<float>>(a, st);
            case kThreeCart: return launch_zero_order_tc<ThreeCart<float>>(a, st);
            case kQuadrotor: return launch_zero_order_tc<Quadrotor<float>>(a, st);
#else
            case kUser: return launch_zero_order_tc<UserSystem<float>>(a, st);
#endif
        }
    }
    switch (system) {
#ifndef IRS_USER_SYSTEM
        case kPendulum: return launch_zero_order<Pendulum<float>, 1>(a, st);
        case kBicycle: return launch_zero_order<Bicycle<float>, 1>(a, st);
        case kThreeCart: return launch_zero_order<ThreeCart<float>, 1>(a, st);
        case kMlp21:
            if (use_mlp_tensor_cores()) return launch_zero_order_mlp<Mlp21<float>>(a, st);
            return launch_zero_order<Mlp21<float>, 1>(a, st);
        case kQuadrotor:
            IRS_REQUIRE(S % 128 == 0, "quadrotor chunk size must be a multiple of 128");
            // 16 regressors: the Gram rows are split over the 4 warps of a block sharing one sample tile
            return launch_zero_order<Quadrotor<float>, 4>(a, st);
#else
        case kUser: return launch_zero_order_user(a, st);
#endif
    }
    set_error("unknown system id %d", system);
    return 1;
}

int irs_smooth_first_order_accumulate(int system, const double* params_host, int nparams, int flags,
                                      const double* x_nom, const double* u_nom, int P, long long N,
                                      const float* sigma_host, const float* noise,
                                      unsigned long long seed, unsigned iter, unsigned stream_id,
                                      unsigned p0, unsigned long long i0,
                                      int C, long long S, float* partials, void* stream) {
    SmoothArgs a;
    IRS_REQUIRE(system != kThreeCart,
                "three_cart is not differentiable and has no Jacobian (three_cart_dynamics.py:20)");
    if (fill_smooth_args(&a, system, params_host, nparams, flags, x_nom, u_nom, P, N, sigma_host, noise,
                         seed, iter, stream_id, p0, i0, C, S, partials))
        return 1;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((long long)P * C);
    switch (system) {
#ifndef IRS_USER_SYSTEM
        case kPendulum:
            g_last_smooth_func = (const void*)smooth_first_order_kernel<Pendulum<float>>;
            smooth_first_order_kernel<Pendulum<float>><<<grid, 128, 0, st>>>(a);
            break;
        case kBicycle:
            g_last_smooth_func = (const void*)smooth_first_order_kernel<Bicycle<float>>;
            smooth_first_order_kernel<Bicycle<float>><<<grid, 128, 0, st>>>(a);
            break;
        case kQuadrotor:
            g_last_smooth_func = (const void*)smooth_first_order_kernel<Quadrotor<float>>;
            smooth_first_order_kernel<Quadrotor<float>><<<grid, 128, 0, st>>>(a);
            break;
        case kMlp21:
            g_last_smooth_func = (const void*)smooth_first_order_kernel<Mlp21<float>>;
            smooth_first_order_kernel<Mlp21<float>><<<grid, 128, 0, st>>>(a);
            break;
#else
        case kUser:
            if constexpr (UserSystem<float>::kHasJacobian) {
                g_last_smooth_func = (const void*)smooth_first_order_kernel<UserSystem<float>>;
                smooth_first_order_kernel<UserSystem<float>><<<grid, 128, 0, st>>>(a);
                break;
            } else {
                set_error("the user system was built without a Jacobian body: no first-order smoothing");
                return 1;
            }
#endif
        default: set_error("unknown system id %d", system); return 1;
    }
    return check_launch("smooth_first_order_kernel");
}

int irs_smooth_reduce_chunks(int system, int order, const float* partials, int P, int C,
                             double* reduced, void* stream) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    IRS_REQUIRE(partials && reduced && P >= 1 && C >= 1, "bad reduce arguments");
    const int width = irs_partial_width(system, order);
    reduce_chunks_kernel<<<grid_for((long long)P * width, 256), 256, 0, (cudaStream_t)stream>>>(
        partials, P, C, width, reduced);
    return check_launch("reduce_chunks_kernel");
}

// Index tables of the finalize kernel (smooth.cuh: constant-initialised __device__ data, per device).
static const FinalizeTables* finalize_tables(int system) {
    const FinalizeTables* base = nullptr;
    if (cudaGetSymbolAddress((void**)&base, g_finalize_tables) != cudaSuccess) return nullptr;
    return base + system;
}

// Blocks of the one-block-per-point finalize kernels that can be resident together on this device.
static int finalize_resident_blocks(int system, int order, int* out) {
    int per_sm = 0;
    cudaError_t e = cudaSuccess;
    if (order == 0) {
        IRS_DISPATCH_SYSTEM(system, double, Sys,
                            (e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(
                                 &per_sm, finalize_zero_order_kernel<Sys, kFinalizeThreads>, kFinalizeThreads, 0)));
    } else {
        switch (system) {
#ifndef IRS_USER_SYSTEM
            case kPendulum: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, finalize_first_order_kernel<Pendulum<double>>, kFinalizeThreads, 0); break;
            case kBicycle: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, finalize_first_order_kernel<Bicycle<double>>, kFinalizeThreads, 0); break;
            case kQuadrotor: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, finalize_first_order_kernel<Quadrotor<double>>, kFinalizeThreads, 0); break;
            case kMlp21: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, finalize_first_order_kernel<Mlp21<double>>, kFinalizeThreads, 0); break;
#else
            case kUser:
                if constexpr (UserSystem<double>::kHasJacobian) {
                    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, finalize_first_order_kernel<UserSystem<double>>, kFinalizeThreads, 0);
                    break;
                } else {
                    set_error("system %d has no first-order path", system);
                    return 1;
                }
#endif
            default: set_error("system %d has no first-order path", system); return 1;
        }
    }
    if (e != cudaSuccess) return check_launch("cudaOccupancyMaxActiveBlocksPerMultiprocessor");
    *out = per_sm * num_sms();
    return 0;
}

static int smooth_finalize_impl(int system, const double* params_host, int nparams, int order,
                                const double* x_nom, const double* u_nom, int P, int C,
                                const float* partials, const double* reduced, int nranks,
                                long long rank_stride, double n_total, int centered,
                                double* At, double* Bt, double* ct, int* status, const PeerFusedArgs* peer,
                                void* stream) {
    FinalizeArgs a;
    if (load_params(system, params_host, nparams, &a.prm)) return 1;
    IRS_REQUIRE(order == 0 || order == 1, "order must be 0 or 1");
    IRS_REQUIRE(x_nom && u_nom && At && Bt && ct && status, "null pointer argument");
    IRS_REQUIRE((partials != nullptr) != (reduced != nullptr),
                "exactly one of partials (fp32 per-chunk) and reduced (fp64) must be given");
    a.reduced = reduced;
    IRS_REQUIRE(P >= 1 && C >= 1 && nranks >= 1 && n_total >= 1.0, "bad finalize arguments");
    IRS_REQUIRE(!(order == 1 && system == kThreeCart), "three_cart has no Jacobian");
    IRS_REQUIRE(!centered || (system == kThreeCart && order == 0), "centred accumulation is built for three_cart only");
    a.centered = centered ? 1 : 0;
    a.x_nom = x_nom;  a.u_nom = u_nom;  a.partials = partials;  a.rank_stride = rank_stride;
    a.R = nranks;  a.P = P;  a.C = C;  a.n_total = n_total;
    a.At = At;  a.Bt = Bt;  a.ct = ct;  a.status = status;
    memset(&a.peer, 0, sizeof(a.peer));
    if (peer != nullptr) a.peer = *peer;
    cudaStream_t st = (cudaStream_t)stream;
    a.tables = finalize_tables(system);
    if (a.tables == nullptr) return check_launch("finalize index tables") ? 1 : (set_error("finalize index tables"), 1);
    // many points: four threads per point, else one block per point (IRS_FINALIZE_VARIANT=block|quad
    // overrides; the variants are bit-identical, tests/test_gpu_parity.py)
    bool quad = P > 8 * num_sms();
    if (const char* e = getenv("IRS_FINALIZE_VARIANT")) {
        if (!strcmp(e, "block")) quad = false;
        else if (!strcmp(e, "quad")) quad = true;
    }
    if (peer != nullptr) quad = false;      // the fused exchange lives in the one-block-per-point kernels
    if (centered) quad = false;             // ... and so does the un-shift of a centred Gram
    if (quad || order == 1) {
        // f(xbar, ubar) in fp64 (scalar dynamics, ...zero_order.py:61) -> ct; the finalize kernel turns it into c
        IRS_DISPATCH_SYSTEM(system, double, Sys,
                            (dyn_batch_kernel<double, Sys><<<grid_for(P, 128), 128, 0, st>>>(a.prm, 0, x_nom, u_nom, ct, P)));
        if (check_launch("nominal dynamics kernel")) return 1;
    }
    const unsigned grid = (unsigned)P;      // one block per nominal point
    if (order == 0) {
        if (quad) {
            IRS_DISPATCH_SYSTEM(system, double, Sys, {
                using QC = FinalizeQuadCfg<Sys>;
                auto kern = finalize_zero_order_quad_kernel<Sys>;
                if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)QC::kSmemBytes) != cudaSuccess)
                    return check_launch("cudaFuncSetAttribute(finalize_zero_order_quad_kernel)");
                kern<<<(unsigned)((P + QC::PPB - 1) / QC::PPB), kFinalizeQuadThreads, QC::kSmemBytes, st>>>(a);
            });
        } else {
            IRS_DISPATCH_SYSTEM(system, double, Sys,
                                (finalize_zero_order_kernel<Sys, kFinalizeThreads><<<grid, kFinalizeThreads, 0, st>>>(a)));
        }
    } else {
        switch (system) {
#ifndef IRS_USER_SYSTEM
            case kPendulum: finalize_first_order_kernel<Pendulum<double>><<<grid, kFinalizeThreads, 0, st>>>(a); break;
            case kBicycle: finalize_first_order_kernel<Bicycle<double>><<<grid, kFinalizeThreads, 0, st>>>(a); break;
            case kQuadrotor: finalize_first_order_kernel<Quadrotor<double>><<<grid, kFinalizeThreads, 0, st>>>(a); break;
            case kMlp21: finalize_first_order_kernel<Mlp21<double>><<<grid, kFinalizeThreads, 0, st>>>(a); break;
#else
            case kUser:
                if constexpr (UserSystem<double>::kHasJacobian) {
                    finalize_first_order_kernel<UserSystem<double>><<<grid, kFinalizeThreads, 0, st>>>(a);
                    break;
                } else {
                    set_error("the user system was built without a Jacobian body: no first-order smoothing");
                    return 1;
                }
#endif
            default: set_error("unknown system id %d", system); return 1;
        }
    }
    return check_launch("finalize_kernel");
}

int irs_smooth_finalize(int system, const double* params_host, int nparams, int order,
                        const double* x_nom, const double* u_nom, int P, int C,
                        const float* partials, const double* reduced, int nranks,
                        long long rank_stride, double n_total, int centered,
                        double* At, double* Bt, double* ct, int* status, void* stream) {
    return smooth_finalize_impl(system, params_host, nparams, order, x_nom, u_nom, P, C, partials, reduced, nranks,
                                rank_stride, n_total, centered, At, Bt, ct, status, nullptr, stream);
}

int irs_smooth_finalize_peer_capacity(int system, int order, int* max_points) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems && (order == 0 || order == 1) && max_points, "bad arguments");
    return finalize_resident_blocks(system, order, max_points);
}

int irs_smooth_finalize_peer(int system, const double* params_host, int nparams, int order,
                             const double* x_nom, const double* u_nom, int P, int C, const float* partials,
                             const void* peer_bufs_dev, const void* peer_flags_dev, int* epoch_dev,
                             unsigned int* done_counter, long long slot_stride, int flag_stride,
                             int rank, int world, double timeout_s, double n_total, int centered,
                             double* At, double* Bt, double* ct, int* status, void* stream) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    IRS_REQUIRE(partials && peer_bufs_dev && peer_flags_dev && epoch_dev && done_counter, "null pointer argument");
    IRS_REQUIRE(world >= 1 && world <= kFinalizeThreads && rank >= 0 && rank < world, "bad rank / world");
    IRS_REQUIRE(timeout_s > 0.0, "timeout must be positive");
    const int width = irs_partial_width(system, order);
    IRS_REQUIRE(slot_stride >= (long long)P * width && flag_stride >= P, "exchange buffers too small for P=%d", P);
    int resident = 0;
    if (finalize_resident_blocks(system, order, &resident)) return 1;
    IRS_REQUIRE(P <= resident, "the fused exchange needs its %d blocks co-resident (%d fit): use the all-gather path", P, resident);
    PeerFusedArgs px{(double* const*)peer_bufs_dev, (int* const*)peer_flags_dev, epoch_dev, done_counter,
                     slot_stride, flag_stride, rank, world, (unsigned long long)(timeout_s * 1e9),
                     kPeerExchange, 0, 0, 0};
    return smooth_finalize_impl(system, params_host, nparams, order, x_nom, u_nom, P, C, partials, nullptr, 1, 0,
                                n_total, centered, At, Bt, ct, status, &px, stream);
}

int irs_smooth_finalize_gather(int system, const double* params_host, int nparams, int order,
                               const double* x_nom, const double* u_nom, int P, int C, const float* partials,
                               const void* peer_out_bufs_dev, const void* peer_flags_dev, int* epoch_dev,
                               unsigned int* done_counter, long long out_stride, int p0, int P_total,
                               int rank, int world, double timeout_s, double n_total, int centered,
                               double* ct_scratch, void* stream) {
    IRS_REQUIRE(system >= 0 && system < kNumSystems, "unknown system id %d", system);
    IRS_REQUIRE(peer_out_bufs_dev && peer_flags_dev && epoch_dev && done_counter, "null pointer argument");
    IRS_REQUIRE(world >= 1 && world <= kFinalizeThreads && rank >= 0 && rank < world, "bad rank / world");
    IRS_REQUIRE(timeout_s > 0.0 && P >= 0 && p0 >= 0 && P_total >= 1 && p0 + P <= P_total, "bad gather arguments");
    const SystemDims dm = system_dims(system);
    IRS_REQUIRE(out_stride >= (long long)P_total * (dm.n * (dm.n + dm.m + 1) + 1), "output buffers too small");
    PeerFusedArgs px{(double* const*)peer_out_bufs_dev, (int* const*)peer_flags_dev, epoch_dev, done_counter,
                     0, 0, rank, world, (unsigned long long)(timeout_s * 1e9), kPeerGather, p0, P_total, out_stride};
    if (P == 0) {      // this rank owns no timestep: it still takes part in the step
        peer_gather_wait_kernel<<<1, 128, 0, (cudaStream_t)stream>>>(px);
        return check_launch("peer_gather_wait_kernel");
    }
    IRS_REQUIRE(partials && ct_scratch, "null pointer argument");
    // the kernel writes its results into the ranks' output buffers; ct_scratch [P, n] is the local scratch
    // the first-order finalize keeps f(xbar, ubar) in; status goes into the gathered buffer too
    return smooth_finalize_impl(system, params_host, nparams, order, x_nom, u_nom, P, C, partials, nullptr, 1, 0,
                                n_total, centered, ct_scratch, ct_scratch, ct_scratch, (int*)ct_scratch, &px, stream);
}

int irs_exact_linearize(int system, const double* params_host, int nparams,
                        const double* x_nom, const double* u_nom, int P,
                        double* At, double* Bt, double* ct, void* stream) {
    SysParams prm;
    if (load_params(system, params_host, nparams, &prm)) return 1;
    IRS_REQUIRE(system != kThreeCart,
                "three_cart is not differentiable and has no Jacobian (three_cart_dynamics.py:20)");
    IRS_REQUIRE(x_nom && u_nom && At && Bt && ct, "null pointer argument");
    IRS_REQUIRE(P >= 1, "need at least one nominal point");
    cudaStream_t st = (cudaStream_t)stream;
    switch (system) {
#ifndef IRS_USER_SYSTEM
        case kPendulum: exact_linearize_kernel<Pendulum<double>><<<(P + 63) / 64, 64, 0, st>>>(prm, x_nom, u_nom, P, At, Bt, ct); break;
        case kBicycle: exact_linearize_kernel<Bicycle<double>><<<(P + 63) / 64, 64, 0, st>>>(prm, x_nom, u_nom, P, At, Bt, ct); break;
        case kQuadrotor: exact_linearize_kernel<Quadrotor<double>><<<(P + 63) / 64, 64, 0, st>>>(prm, x_nom, u_nom, P, At, Bt, ct); break;
        case kMlp21: exact_linearize_kernel<Mlp21<double>><<<(P + 63) / 64, 64, 0, st>>>(prm, x_nom, u_nom, P, At, Bt, ct); break;
#else
        case kUser:
            if constexpr (UserSystem<double>::kHasJacobian) {
                exact_linearize_kernel<UserSystem<double>><<<(P + 63) / 64, 64, 0, st>>>(prm, x_nom, u_nom, P, At, Bt, ct);
                break;
            } else {
                set_error("the user system was built without a Jacobian body: no exact linearization");
                return 1;
            }
#endif
        default: set_error("unknown system id %d", system); return 1;
    }
    return check_launch("exact_linearize_kernel");
}

int irs_mlp_register(int dim_x, int dim_u, int h1, int h2, const float* W1, const float* b1, const float* W2,
                     const float* b2, const float* W3, const float* b3, int* handle) {
    IRS_REQUIRE(W1 && b1 && W2 && b2 && W3 && b3 && handle, "null pointer argument");
    IRS_REQUIRE(dim_x >= 1 && dim_u >= 1, "need dim_x >= 1 and dim_u >= 1");
    IRS_REQUIRE(h1 >= 1 && h1 <= kMlpMaxHidden && h2 >= 1 && h2 <= kMlpMaxHidden,
                "hidden widths must lie in [1, %d], got %d and %d", kMlpMaxHidden, h1, h2);
    const int d = dim_x + dim_u, n = dim_x;
    const long long count = MlpView::floats(d, n, h1, h2);
    std::vector<float> host((size_t)count);
    MlpView v(host.data(), d, n, h1, h2);
    memcpy(const_cast<float*>(v.w1), W1, sizeof(float) * h1 * d);
    memcpy(const_cast<float*>(v.b1), b1, sizeof(float) * h1);
    memcpy(const_cast<float*>(v.w2), W2, sizeof(float) * h2 * h1);
    memcpy(const_cast<float*>(v.b2), b2, sizeof(float) * h2);
    memcpy(const_cast<float*>(v.w3), W3, sizeof(float) * n * h2);
    memcpy(const_cast<float*>(v.b3), b3, sizeof(float) * n);
    for (int j = 0; j < h2; ++j)
        for (int q = 0; q < h1; ++q) const_cast<float*>(v.w2t)[(size_t)q * h2 + j] = W2[(size_t)j * h1 + q];
    for (float x : host) IRS_REQUIRE(x == x && x - x == 0.f, "network weights must be finite");
    // hidden layer as tensor-core operand: B[j][k] = W2[j][k] (k < h1), b2[j] (k = h1), zero padding; two bf16
    // pieces, round to nearest even, hi + lo = the float32 weight to 2^-17 relative
    const MlpTcLayout L(h1, h2);
    std::vector<unsigned short> tc((size_t)L.blob_bytes() / 2, 0);     // [W2 hi | W2 lo | B1 hi | B1 lo] bf16 elements
    auto bf16_rn = [](float x) -> unsigned short {
        uint32_t u;
        memcpy(&u, &x, 4);
        u += 0x7fffu + ((u >> 16) & 1u);
        return (unsigned short)(u >> 16);
    };
    auto bf16_float = [](unsigned short h) -> float {
        const uint32_t u = (uint32_t)h << 16;
        float f;
        memcpy(&f, &u, 4);
        return f;
    };
    for (int j = 0; j < h2; ++j)
        for (int k = 0; k <= h1; ++k) {
            const float wv = k < h1 ? W2[(size_t)j * h1 + k] : b2[j];
            const unsigned short hi = bf16_rn(wv), lo = bf16_rn(wv - bf16_float(hi));
            const size_t at = (size_t)L.b_offset(j, k) / 2;
            tc[at] = hi;
            tc[(size_t)L.b_piece_bytes() / 2 + at] = lo;
        }
    // first layer as operand: row j = (W1[j][0..d), b1[j], 0..), row h1 = (0, .., 0, 1): the constant unit
    IRS_REQUIRE(d + 1 <= 8, "the first layer takes at most 7 inputs");
    {
        const size_t base_hi = (size_t)L.b_piece_bytes(), base_lo = base_hi + (size_t)L.b1_piece_bytes() / 2;
        for (int j = 0; j <= h1; ++j)
            for (int k = 0; k <= d; ++k) {
                const float wv = j < h1 ? (k < d ? W1[(size_t)j * d + k] : b1[j]) : (k == d ? 1.f : 0.f);
                const unsigned short hi = bf16_rn(wv), lo = bf16_rn(wv - bf16_float(hi));
                const size_t at = (size_t)L.b1_offset(j, k) / 2;
                tc[base_hi + at] = hi;
                tc[base_lo + at] = lo;
            }
    }
    MlpEntry e{nullptr, nullptr, d, n, h1, h2, 0};
    cudaGetDevice(&e.device);
    if (cudaMalloc(&e.blob, sizeof(float) * count) != cudaSuccess) return check_launch("cudaMalloc(network)");
    if (cudaMalloc(&e.w2_tc, sizeof(unsigned short) * tc.size()) != cudaSuccess) {
        cudaFree(e.blob);
        return check_launch("cudaMalloc(network operand)");
    }
    if (cudaMemcpy(e.blob, host.data(), sizeof(float) * count, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(e.w2_tc, tc.data(), sizeof(unsigned short) * tc.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(e.blob);
        cudaFree(e.w2_tc);
        return check_launch("cudaMemcpy(network)");
    }
    std::lock_guard<std::mutex> lock(g_mlp_mutex);
    g_mlps.push_back(e);
    *handle = (int)g_mlps.size() - 1;
    return 0;
}

int irs_mlp_release(int handle) {
    std::lock_guard<std::mutex> lock(g_mlp_mutex);
    IRS_REQUIRE(handle >= 0 && handle < (int)g_mlps.size() && g_mlps[handle].blob != nullptr,
                "unknown network handle %d", handle);
    cudaFree(g_mlps[handle].blob);      // synchronises with the device: no kernel still reads it
    cudaFree(g_mlps[handle].w2_tc);
    g_mlps[handle].blob = nullptr;
    g_mlps[handle].w2_tc = nullptr;
    return 0;
}

int irs_philox_dump(int P, long long N, int d, const float* sigma_host, unsigned long long seed,
                    unsigned iter, unsigned stream_id, unsigned p0, unsigned long long i0, int antithetic,
                    unsigned* words, float* deltas, void* stream) {
    IRS_REQUIRE(P >= 1 && N >= 1 && d >= 1 && d <= kMaxRegressors, "bad dump arguments");
    IRS_REQUIRE(deltas == nullptr || sigma_host != nullptr, "deltas need sigma");
    PhiloxDumpArgs a;
    a.P = P;  a.d = d;  a.N = N;
    a.seed_lo = (uint32_t)(seed & 0xffffffffull);  a.seed_hi = (uint32_t)(seed >> 32);
    a.iter = iter;  a.stream = stream_id;  a.p0 = p0;  a.i0 = i0;  a.antithetic = antithetic ? 1 : 0;
    a.words = words;  a.deltas = deltas;
    for (int c = 0; c < kMaxRegressors; ++c)
        a.sigma_scaled[c] = (sigma_host != nullptr && c < d) ? kBoxMullerScale * sigma_host[c] : 0.f;
    const long long total = (long long)P * N * ((d + 3) / 4);
    philox_dump_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(a);
    return check_launch("philox_dump_kernel");
}

int irs_dynamics_batch_f32(int system, const double* params_host, int nparams, int batch_variant,
                           const float* x, const float* u, float* out, long long B, void* stream) {
    return dynamics_batch_impl<float>(system, params_host, nparams, batch_variant, x, u, out, B, stream);
}
int irs_dynamics_batch_f64(int system, const double* params_host, int nparams, int batch_variant,
                           const double* x, const double* u, double* out, long long B, void* stream) {
    return dynamics_batch_impl<double>(system, params_host, nparams, batch_variant, x, u, out, B, stream);
}
int irs_jacobian_xu_batch_f32(int system, const double* params_host, int nparams,
                              const float* x, const float* u, float* J, long long B, void* stream) {
    return jacobian_batch_impl<float>(system, params_host, nparams, x, u, J, B, stream);
}
int irs_jacobian_xu_batch_f64(int system, const double* params_host, int nparams,
                              const double* x, const double* u, double* J, long long B, void* stream) {
    return jacobian_batch_impl<double>(system, params_host, nparams, x, u, J, B, stream);
}

int irs_project_batch_f64(int system, const double* params_host, int nparams, double* x,
                          long long B, void* stream) {
    SysParams prm;
    if (load_params(system, params_host, nparams, &prm)) return 1;
    IRS_REQUIRE(B >= 0, "negative batch");
    if (B == 0) return 0;
    IRS_REQUIRE(x != nullptr, "null pointer argument");
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_SYSTEM(system, double, Sys,
                        (project_batch_kernel<double, Sys><<<grid_for(B, 128), 128, 0, st>>>(prm, x, B)));
    return check_launch("project_batch_kernel");
}

static int tvlqr_riccati_impl(int n, int m, const double* At, const double* Bt, const double* ct,
                              const double* Q, const double* Qd, const double* R,
                              const double* xd, long long xd_stride, int I, int T,
                              double* K, double* k, int* status, double* Hinv_out, double* P_out, void* stream,
                              int t_lo = 0, int t_hi = 0, double* carry = nullptr) {
    IRS_REQUIRE(At && Bt && ct && Q && Qd && R && xd && K && k && status, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    TvlqrArgs a{At, Bt, ct, Q, Qd, R, xd, xd_stride, K, k, status, I, T, Hinv_out, P_out, t_lo, t_hi, carry};
    if (t_hi > 0) {      // a segment of the recursion: register-tiled kernel only
        IRS_REQUIRE(0 <= t_lo && t_lo < t_hi && t_hi <= T, "bad segment [%d, %d) of T=%d", t_lo, t_hi, T);
        IRS_REQUIRE(n % 2 == 0 && m % 2 == 0 && Hinv_out == nullptr && P_out == nullptr,
                    "segmented Riccati needs even n, m (n=%d, m=%d)", n, m);
        IRS_REQUIRE((t_lo == 0 && t_hi == T) || carry != nullptr, "a partial segment needs the carry buffer");
    }
#if defined(IRS_USER_SYSTEM) && !IRS_USER_BUILTIN_DIMS
    IRS_REQUIRE(t_hi == 0, "segmented Riccati is not built for n=%d m=%d", n, m);
    return irs_tvlqr_riccati_any(n, m, At, Bt, ct, Q, Qd, R, xd, xd_stride, I, T, K, k, status, Hinv_out, P_out, stream);
#else
    cudaStream_t st = (cudaStream_t)stream;
    // few instances: one block per instance (latency); many: one warp per instance (throughput) —
    // except where the register-tiled block kernel applies (even n, m): it moves half the shared-memory
    // bytes per DFMA and is the faster one at every instance count (4096 quadrotor instances: 1.30 ms
    // against 1.63 ms), so those dimensions always take it and a problem's result does not depend on I
    const bool tiled_dims = n % 2 == 0 && m % 2 == 0 && Hinv_out == nullptr && P_out == nullptr;
    bool per_block = I <= 2 * num_sms() || tiled_dims;
    if (const char* e = getenv("IRS_TVLQR_VARIANT")) {      // tuning / tests: block | warp
        if (!strcmp(e, "block")) per_block = true;
        else if (!strcmp(e, "warp")) per_block = false;
    }
    if (t_hi > 0) per_block = true;                                 // segments exist in the tiled kernel only
    const bool extra = Hinv_out != nullptr || P_out != nullptr;     // only the generic kernel writes them
    // many instances of a 4-divisible problem (quadrotor): two instances per warp, 4 x 4 register tiles
    // (tvlqr.cuh: tvlqr_riccati_packed_kernel).  That kernel's time is flat up to one block of eight instances per
    // SM (0.37 ms at T = 100 up to 1,184 instances, then 0.49 / 0.64 / 0.83 ms at 2048 / 3072 / 4096); the block
    // kernel takes 0.19 / 0.23 / 0.30 / 0.47 / 0.71 / 1.28 ms at 300 / 512 / 768 / 1024 / 2048 / 4096 and crosses it
    // between 768 and 1024 instances (measured with tools/batched_bench.py).  Results of the two kernels agree to
    // 1e-10 (summation order), so a shard of 512 instances and the unsharded 4096 differ at that level.
    // IRS_TVLQR_VARIANT=block|warp|packed overrides.
    constexpr long long kPackedMinInstances = 1000;
    const char* variant = getenv("IRS_TVLQR_VARIANT");
    const bool force_packed = variant != nullptr && !strcmp(variant, "packed");
#if !defined(IRS_USER_SYSTEM) || (IRS_USER_N == 12 && IRS_USER_M == 4)
    if (n == 12 && m == 4 && !extra && t_hi == 0 && (force_packed || (variant == nullptr && I >= kPackedMinInstances))) {
        auto kern = tvlqr_riccati_packed_kernel<12, 4>;
        const int smem = (int)sizeof(RicPackSmem<12, 4>);
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess)
            return check_launch("cudaFuncSetAttribute(tvlqr_riccati_packed_kernel)");
        kern<<<(unsigned)((I + kRicPackPerBlock - 1) / kRicPackPerBlock), kRicPackThreads, smem, st>>>(a);
        return check_launch("tvlqr_riccati_packed_kernel");
    }
#else
    (void)force_packed;
#endif
    IRS_DISPATCH_DIMS(n, m, {
        if (per_block) {
            if constexpr (N_ % 2 == 0 && M_ % 2 == 0) {
                if (!extra) {
                    tvlqr_riccati_tiled_kernel<N_, M_>
                        <<<(unsigned)I, kTvlqrTiledThreads, sizeof(TvlqrTiledSmem<N_, M_>), st>>>(a);
                    return check_launch("tvlqr_riccati_tiled_kernel");
                }
            }
            tvlqr_riccati_kernel<N_, M_, kTvlqrBlockThreads>
                <<<(unsigned)I, kTvlqrBlockThreads, sizeof(TvlqrSmem<N_, M_>), st>>>(a);
        } else {
            const unsigned grid = (unsigned)((I + kTvlqrWarps - 1) / kTvlqrWarps);
            tvlqr_riccati_kernel<N_, M_, 32><<<grid, 32 * kTvlqrWarps, sizeof(TvlqrSmem<N_, M_>) * kTvlqrWarps, st>>>(a);
        }
    });
    return check_launch("tvlqr_riccati_kernel");
#endif
}

int irs_tvlqr_riccati(int n, int m, const double* At, const double* Bt, const double* ct,
                      const double* Q, const double* Qd, const double* R,
                      const double* xd, long long xd_stride, int I, int T,
                      double* K, double* k, int* status, void* stream) {
    return tvlqr_riccati_impl(n, m, At, Bt, ct, Q, Qd, R, xd, xd_stride, I, T, K, k, status, nullptr, nullptr, stream);
}

int irs_tvlqr_riccati_segment(int n, int m, const double* At, const double* Bt, const double* ct,
                              const double* Q, const double* Qd, const double* R,
                              const double* xd, long long xd_stride, int I, int T, int t_lo, int t_hi,
                              double* carry, double* K, double* k, int* status, void* stream) {
    IRS_REQUIRE(t_hi >= 1, "need t_hi >= 1");
    return tvlqr_riccati_impl(n, m, At, Bt, ct, Q, Qd, R, xd, xd_stride, I, T, K, k, status, nullptr, nullptr, stream,
                              t_lo, t_hi, carry);
}

int irs_tvlqr_riccati_ex(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* Q, const double* Qd, const double* R,
                         const double* xd, long long xd_stride, int I, int T,
                         double* K, double* k, int* status, double* Hinv_out, double* P_out, void* stream) {
    return tvlqr_riccati_impl(n, m, At, Bt, ct, Q, Qd, R, xd, xd_stride, I, T, K, k, status, Hinv_out, P_out, stream);
}

int irs_tvlqr_plan_rows(int n, int m, const double* At, const double* Bt, const double* ct,
                        const double* K, const double* k, int I, int T, double* scratch, void* stream) {
    IRS_REQUIRE(At && Bt && ct && K && k && scratch, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1 && I <= 65535, "need 1 <= I <= 65535 and T >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    PlanCheckArgs a{At, Bt, ct, K, k, nullptr, nullptr, nullptr, nullptr, nullptr, 0.0, nullptr, scratch, I, T};
    IRS_DISPATCH_DIMS(n, m, { plan_rows_kernel<N_, M_><<<dim3((unsigned)T, (unsigned)I), 32, 0, st>>>(a); });
    return check_launch("plan_rows_kernel");
}

int irs_tvlqr_plan_check(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* K, const double* k, const double* x_trj,
                         const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                         double tol, int I, int T, int rows_ready, int* violated, double* scratch, void* stream) {
    IRS_REQUIRE(At && Bt && ct && K && k && x_trj && xlo && xhi && ulo && uhi && violated && scratch,
                "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1 && I <= 65535, "need 1 <= I <= 65535 and T >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemsetAsync(violated, 0, sizeof(int) * I, st) != cudaSuccess) return check_launch("cudaMemsetAsync");
    PlanCheckArgs a{At, Bt, ct, K, k, x_trj, xlo, xhi, ulo, uhi, tol, violated, scratch, I, T};
    IRS_DISPATCH_DIMS(n, m, {
        // rows_ready: irs_tvlqr_plan_rows has filled `scratch` already (it needs the gains only, so a caller
        // can run it beside the closed-loop rollout)
        if (!rows_ready) plan_rows_kernel<N_, M_><<<dim3((unsigned)T, (unsigned)I), 32, 0, st>>>(a);
        plan_check_kernel<N_, M_><<<dim3((unsigned)T, (unsigned)I), 32, 0, st>>>(a);
    });
    return check_launch("plan_check_kernel");
}

int irs_tvlqr_box_solve(int system, const double* params_host, int nparams, int mpc,
                        const double* At, const double* Bt, const double* ct,
                        const double* K, const double* Hinv, const double* P,
                        const double* Q, const double* Qd, const double* R,
                        const double* xd, long long xd_stride, const double* dx, const double* du,
                        const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                        long long xbox_stride, long long ubox_stride,
                        const double* x0, const double* K0, const double* k0, double tol,
                        double alpha, double eps, int max_iter, int I, int T,
                        double* x_trj, double* u_trj, double* cost, int* status, int* iters, void* stream) {
    BoxMpcArgs a;
    if (load_params(system, params_host, nparams, &a.prm)) return 1;
    IRS_REQUIRE(At && Bt && ct && K && Hinv && P && Q && Qd && R && xd && dx && du && xlo && xhi && ulo && uhi &&
                    x0 && x_trj && u_trj && cost && status && iters, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1 && max_iter >= 1, "need I >= 1, T >= 1, max_iter >= 1");
    IRS_REQUIRE(alpha > 0.0 && alpha < 2.0 && eps > 0.0, "need 0 < alpha < 2 and eps > 0");
    {
        const SystemDims dm = system_dims(system);
        IRS_REQUIRE((xbox_stride == 0 || xbox_stride == dm.n) && (ubox_stride == 0 || ubox_stride == dm.m),
                    "box strides must be 0 (constant box) or n / m (one box per timestep)");
    }
    a.At = At;  a.Bt = Bt;  a.ct = ct;  a.K = K;  a.Hinv = Hinv;  a.P = P;  a.Q = Q;  a.Qd = Qd;  a.R = R;
    a.xd = xd;  a.xd_stride = xd_stride;  a.dx = dx;  a.du = du;  a.xlo = xlo;  a.xhi = xhi;  a.ulo = ulo;
    a.uhi = uhi;  a.xbox_stride = xbox_stride;  a.ubox_stride = ubox_stride;  a.x0 = x0;  a.K0 = K0;  a.k0 = k0;  a.tol = tol;  a.alpha = alpha;  a.eps = eps;  a.max_iter = max_iter;  a.mpc = mpc ? 1 : 0;
    a.x_trj = x_trj;  a.u_trj = u_trj;  a.cost = cost;  a.status = status;  a.iters = iters;  a.I = I;  a.T = T;
    cudaStream_t st = (cudaStream_t)stream;
    switch (system) {
#ifndef IRS_USER_SYSTEM
        case kPendulum: return launch_box_mpc<Pendulum<double>>(a, st);
        case kBicycle: return launch_box_mpc<Bicycle<double>>(a, st);
        case kQuadrotor: return launch_box_mpc<Quadrotor<double>>(a, st);
        case kThreeCart: return launch_box_mpc<ThreeCart<double>>(a, st);
        case kMlp21: return launch_box_mpc<Mlp21<double>>(a, st);
#else
        case kUser: return launch_box_mpc<UserSystem<double>>(a, st);
#endif
    }
    set_error("unknown system id %d", system);
    return 1;
}

int irs_tvlqr_linear_rollout(int n, int m, const double* At, const double* Bt, const double* ct,
                             const double* K, const double* k, const double* x0, int I, int T,
                             double* xs, double* us, void* stream) {
    IRS_REQUIRE(At && Bt && ct && K && k && x0 && xs && us, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
#if defined(IRS_USER_SYSTEM) && !IRS_USER_BUILTIN_DIMS
    return irs_tvlqr_linear_rollout_any(n, m, At, Bt, ct, K, k, x0, I, T, xs, us, stream);
#else
    TvlqrArgs a{At, Bt, ct, nullptr, nullptr, nullptr, nullptr, 0, const_cast<double*>(K),
                const_cast<double*>(k), nullptr, I, T};
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_DIMS(n, m, (linear_rollout_kernel<N_, M_><<<(I + 63) / 64, 64, 0, st>>>(a, x0, xs, us)));
    return check_launch("linear_rollout_kernel");
#endif
}

// ---- run-time dimensions (tvlqr_any.cuh): every (n, m) up to kTvlqrAnyMaxDim, the built-in pairs included ----
int irs_tvlqr_any_limits(int* max_n, int* max_m) {
    IRS_REQUIRE(max_n && max_m, "null pointer argument");
    *max_n = kTvlqrAnyMaxDim;
    *max_m = kTvlqrAnyMaxDim;
    return 0;
}

#define IRS_REQUIRE_ANY_DIMS(n, m)                                                                  \
    IRS_REQUIRE(n >= 1 && n <= kTvlqrAnyMaxDim && m >= 1 && m <= kTvlqrAnyMaxDim,                   \
                "TVLQR dims n=%d m=%d out of range: need 1 <= n, m <= %d", n, m, kTvlqrAnyMaxDim)

int irs_tvlqr_riccati_any(int n, int m, const double* At, const double* Bt, const double* ct,
                          const double* Q, const double* Qd, const double* R,
                          const double* xd, long long xd_stride, int I, int T,
                          double* K, double* k, int* status, double* Hinv_out, double* P_out, void* stream) {
    IRS_REQUIRE_ANY_DIMS(n, m);
    IRS_REQUIRE(At && Bt && ct && Q && Qd && R && xd && K && k && status, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    IRS_REQUIRE(xd_stride >= 0, "need xd_stride >= 0");
    TvlqrAnyArgs a{TvlqrArgs{At, Bt, ct, Q, Qd, R, xd, xd_stride, K, k, status, I, T, Hinv_out, P_out, 0, 0, nullptr},
                   n, m};
    const size_t smem = tvlqr_riccati_any_smem_bytes(n, m);      // 109 KiB at n = m = 32
    if (cudaFuncSetAttribute(tvlqr_riccati_any_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) !=
        cudaSuccess)
        return check_launch("cudaFuncSetAttribute(tvlqr_riccati_any_kernel)");
    tvlqr_riccati_any_kernel<<<(unsigned)I, tvlqr_any_threads(n, m), smem, (cudaStream_t)stream>>>(a);
    return check_launch("tvlqr_riccati_any_kernel");
}

int irs_tvlqr_linear_rollout_any(int n, int m, const double* At, const double* Bt, const double* ct,
                                 const double* K, const double* k, const double* x0, int I, int T,
                                 double* xs, double* us, void* stream) {
    IRS_REQUIRE_ANY_DIMS(n, m);
    IRS_REQUIRE(At && Bt && ct && K && k && x0 && xs && us, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    TvlqrArgs a{At, Bt, ct, nullptr, nullptr, nullptr, nullptr, 0, const_cast<double*>(K),
                const_cast<double*>(k), nullptr, I, T};
    linear_rollout_any_kernel<<<(unsigned)((I + kRolloutAnyWarps - 1) / kRolloutAnyWarps), 32 * kRolloutAnyWarps, 0,
                                (cudaStream_t)stream>>>(a, n, m, x0, xs, us);
    return check_launch("linear_rollout_any_kernel");
}

int irs_tvlqr_box_qp_any(int n, int m, const double* At, const double* Bt, const double* ct,
                         const double* K, const double* Hinv, const double* P,
                         const double* Q, const double* Qd, const double* R,
                         const double* xd, long long xd_stride, const double* dx, const double* du,
                         const double* xlo, const double* xhi, const double* ulo, const double* uhi,
                         long long xbox_stride, long long ubox_stride, const double* x0,
                         double alpha, double eps, int max_iter, int I, int T,
                         double* x_trj, double* u_trj, int* status, int* iters, void* stream) {
    IRS_REQUIRE_ANY_DIMS(n, m);
    IRS_REQUIRE(At && Bt && ct && K && Hinv && P && Q && Qd && R && xd && dx && du && xlo && xhi && ulo && uhi &&
                    x0 && x_trj && u_trj && status && iters, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1 && max_iter >= 1, "need I >= 1, T >= 1, max_iter >= 1");
    IRS_REQUIRE(xd_stride >= 0, "need xd_stride >= 0");
    IRS_REQUIRE(alpha > 0.0 && alpha < 2.0 && eps > 0.0, "need 0 < alpha < 2 and eps > 0");
    IRS_REQUIRE((xbox_stride == 0 || xbox_stride == n) && (ubox_stride == 0 || ubox_stride == m),
                "box strides must be 0 (constant box) or n / m (one box per timestep)");
    // the ADMM state stays in shared memory under the limit of launch_box_mpc; the per-step matrices join it
    // when they fit too
    constexpr size_t kLimit = 200 * 1024;
    const size_t with_cache = box_qp_any_smem_bytes(n, m, T, true);
    const bool cache = with_cache <= kLimit;
    const size_t smem = cache ? with_cache : box_qp_any_smem_bytes(n, m, T, false);
    if (smem > kLimit) {
        int t_max = 0;
        while (box_qp_any_smem_bytes(n, m, t_max + 1, false) <= kLimit) ++t_max;
        set_error("horizon T=%d too long for the shared-memory resident ADMM state at n=%d m=%d: "
                  "the longest is T=%d (%zu bytes of shared memory at most)", T, n, m, t_max, kLimit);
        return 1;
    }
    BoxQpAnyArgs a{At, Bt, ct, K, Hinv, P, Q, Qd, xd, xd_stride, dx, du, xlo, xhi, ulo, uhi, xbox_stride,
                   ubox_stride, x0, alpha, eps, max_iter, x_trj, u_trj, status, iters, I, T, n, m};
    (void)R;      // the ADMM step only needs the augmented matrices; R is part of the problem's description
    cudaStream_t st = (cudaStream_t)stream;
    auto kern = cache ? box_qp_any_kernel<true> : box_qp_any_kernel<false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess)
        return check_launch("cudaFuncSetAttribute(box_qp_any_kernel)");
    kern<<<(unsigned)I, 32, smem, st>>>(a);
    return check_launch("box_qp_any_kernel");
}

int irs_rollout_closed_loop(int system, const double* params_host, int nparams,
                            const double* K, const double* k, const double* x0,
                            const double* xd, long long xd_stride, const double* Q, const double* R,
                            int I, int T, double* x_trj, double* u_trj, double* cost, void* stream) {
    RolloutArgs a;
    if (load_params(system, params_host, nparams, &a.prm)) return 1;
    IRS_REQUIRE(K && k && x0 && xd && Q && R && x_trj && u_trj && cost, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    a.K = K;  a.k = k;  a.x0 = x0;  a.u_in = nullptr;  a.xd = xd;  a.xd_stride = xd_stride;
    a.Q = Q;  a.R = R;  a.x_trj = x_trj;  a.u_trj = u_trj;  a.cost = cost;  a.I = I;  a.T = T;
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_SYSTEM(system, double, Sys, launch_rollout<Sys, true>(a, st));
    return check_launch("rollout_kernel<closed>");
}

int irs_rollout_open_loop(int system, const double* params_host, int nparams,
                          const double* u_in, const double* x0,
                          const double* xd, long long xd_stride, const double* Q, const double* R,
                          int I, int T, double* x_trj, double* cost, void* stream) {
    RolloutArgs a;
    if (load_params(system, params_host, nparams, &a.prm)) return 1;
    IRS_REQUIRE(u_in && x0 && xd && Q && R && x_trj && cost, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    a.K = nullptr;  a.k = nullptr;  a.x0 = x0;  a.u_in = u_in;  a.xd = xd;  a.xd_stride = xd_stride;
    a.Q = Q;  a.R = R;  a.x_trj = x_trj;  a.u_trj = nullptr;  a.cost = cost;  a.I = I;  a.T = T;
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_SYSTEM(system, double, Sys, launch_rollout<Sys, false>(a, st));
    return check_launch("rollout_kernel<open>");
}

int irs_cem_refit(const double* cost, const double* u_candidates, int B, int T, int m, int n_elite,
                  int* elite, double* mean, double* std_out, void* stream) {
    IRS_REQUIRE(cost && u_candidates && elite && mean && std_out, "null pointer argument");
    IRS_REQUIRE(B >= 1 && T >= 1 && m >= 1 && n_elite >= 1 && n_elite <= B, "need 1 <= n_elite <= B and T, m >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    cem_rank_kernel<<<(B + 255) / 256, 256, 0, st>>>(cost, B, n_elite, elite);
    if (check_launch("cem_rank_kernel")) return 1;
    const int width = T * m;
    cem_refit_kernel<<<(width + 127) / 128, 128, 0, st>>>(u_candidates, elite, B, width, n_elite, mean, std_out);
    return check_launch("cem_refit_kernel");
}

int irs_gram_block_f64(int n, int m, const double* Z, const double* F, long long N, double* out, void* stream) {
    IRS_REQUIRE(Z && F && out, "null pointer argument");
    IRS_REQUIRE(n >= 1 && m >= 0 && n + m <= kMaxRegressors && N >= 1, "bad dimensions");
    const int d = n + m, nacc = gram_nacc(n, m);
    gram_block_f64_kernel<<<(nacc + 127) / 128, 128, 0, (cudaStream_t)stream>>>(Z, F, N, n, d, out);
    return check_launch("gram_block_f64_kernel");
}

int irs_fp32_fma_peak(int iters, float* out, long long out_len, double* flops_host, void* stream) {
    const int blocks = 148 * 8, threads = 256;
    IRS_REQUIRE(out != nullptr && out_len >= (long long)blocks * threads, "scratch buffer too small");
    IRS_REQUIRE(iters >= 1, "iters must be positive");
    fma_peak_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(out, iters, 0.999999f, 1e-6f);
    if (flops_host) *flops_host = 2.0 * 8.0 * (double)iters * blocks * threads;
    return check_launch("fma_peak_kernel");
}

int irs_evaluate_cost(int n, int m, const double* x_trj, const double* u_trj,
                      const double* xd, long long xd_stride, const double* Q, const double* R,
                      int I, int T, double* cost, void* stream) {
    IRS_REQUIRE(x_trj && u_trj && xd && Q && R && cost, "null pointer argument");
    IRS_REQUIRE(I >= 1 && T >= 1, "need I >= 1 and T >= 1");
    cudaStream_t st = (cudaStream_t)stream;
    IRS_DISPATCH_DIMS(n, m, (evaluate_cost_kernel<N_, M_><<<(I + 3) / 4, 128, 0, st>>>(
                                x_trj, u_trj, xd, xd_stride, Q, R, I, T, cost)));
    return check_launch("evaluate_cost_kernel");
}

// ------------------------------------------------------------------------------------------------
// CUDA-graph replay of a fixed call sequence (one iRS-LQR descent, or one linearization with its
// host<->device copies).  Everything submitted to `stream` between irs_graph_begin and
// irs_graph_end — entry points of this library and plain cudaMemcpyAsync alike — becomes one
// graph; irs_graph_update_smoothing rewrites the arguments of the captured accumulate kernel
// (seed, iteration, sigma change between replays; pointers and shapes must not).
// ------------------------------------------------------------------------------------------------
constexpr int kMaxSmoothNodes = 16;      // accumulate launches per captured sequence (timestep segments)
struct IrsGraph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int num_smooth = 0;
    cudaGraphNode_t smooth_node[kMaxSmoothNodes] = {};
    cudaKernelNodeParams smooth_params[kMaxSmoothNodes] = {};
    SmoothArgs args[kMaxSmoothNodes] = {};
};

int irs_graph_begin(void* stream) {
    g_last_smooth_func = nullptr;
    if (cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess)
        return check_launch("cudaStreamBeginCapture");
    return 0;
}

int irs_graph_end(void* stream, void** graph_out) {
    IRS_REQUIRE(graph_out != nullptr, "null pointer argument");
    IrsGraph* g = new IrsGraph();
    if (cudaStreamEndCapture((cudaStream_t)stream, &g->graph) != cudaSuccess || g->graph == nullptr) {
        delete g;
        return check_launch("cudaStreamEndCapture") ? 1 : (set_error("stream capture produced no graph"), 1);
    }
    // locate the accumulate kernel node
    size_t nn = 0;
    cudaGraphGetNodes(g->graph, nullptr, &nn);
    cudaGraphNode_t* nodes = new cudaGraphNode_t[nn ? nn : 1];
    cudaGraphGetNodes(g->graph, nodes, &nn);
    for (size_t i = 0; i < nn && g_last_smooth_func != nullptr; ++i) {
        cudaGraphNodeType ty;
        if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp;
        if (cudaGraphKernelNodeGetParams(nodes[i], &kp) != cudaSuccess) continue;
        if (kp.func == g_last_smooth_func && g->num_smooth < kMaxSmoothNodes) {
            const int q = g->num_smooth++;
            g->smooth_node[q] = nodes[i];
            g->smooth_params[q] = kp;
            g->args[q] = *reinterpret_cast<const SmoothArgs*>(kp.kernelParams[0]);
        }
    }
    delete[] nodes;
    cudaGetLastError();
    if (cudaGraphInstantiate(&g->exec, g->graph, 0) != cudaSuccess) {
        const int rc = check_launch("cudaGraphInstantiate");
        cudaGraphDestroy(g->graph);
        delete g;
        return rc ? rc : 1;
    }
    *graph_out = g;
    return 0;
}

int irs_graph_update_smoothing(void* graph, const float* sigma_host, unsigned long long seed, unsigned iter,
                               unsigned stream_id) {
    IrsGraph* g = reinterpret_cast<IrsGraph*>(graph);
    IRS_REQUIRE(g != nullptr && g->exec != nullptr, "invalid graph handle");
    IRS_REQUIRE(g->num_smooth > 0, "the captured sequence contains no smoothing accumulate kernel");
    IRS_REQUIRE(iter < (1u << 24), "iter out of range");
    for (int q = 0; q < g->num_smooth; ++q) {      // every accumulate launch of the sequence (timestep segments)
        SmoothArgs& a = g->args[q];
        a.seed_lo = (uint32_t)(seed & 0xffffffffull);
        a.seed_hi = (uint32_t)(seed >> 32);
        a.iter = iter;
        a.stream = stream_id;
        if (sigma_host != nullptr) {
            // sigma holds n + m entries; the remaining slots stay zero as in fill_smooth_args
            for (int c = 0; c < a.nreg && c < kMaxRegressors; ++c) a.sigma_scaled[c] = kBoxMullerScale * sigma_host[c];
        }
        void* arg_ptrs[1] = {&a};
        cudaKernelNodeParams kp = g->smooth_params[q];
        kp.kernelParams = arg_ptrs;
        kp.extra = nullptr;
        if (cudaGraphExecKernelNodeSetParams(g->exec, g->smooth_node[q], &kp) != cudaSuccess)
            return check_launch("cudaGraphExecKernelNodeSetParams");
    }
    return 0;
}

int irs_graph_launch(void* graph, void* stream) {
    IrsGraph* g = reinterpret_cast<IrsGraph*>(graph);
    IRS_REQUIRE(g != nullptr && g->exec != nullptr, "invalid graph handle");
    if (cudaGraphLaunch(g->exec, (cudaStream_t)stream) != cudaSuccess) return check_launch("cudaGraphLaunch");
    return 0;
}

int irs_graph_destroy(void* graph) {
    IrsGraph* g = reinterpret_cast<IrsGraph*>(graph);
    if (g == nullptr) return 0;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return 0;
}

}  // extern "C"
