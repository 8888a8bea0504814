// Zero-order smoothing with the Gram accumulation on the 5th-generation tensor cores (tcgen05).
//
// Per sample the fit needs the rank-1 update  [dx du]^T [dx du | dF]  (d x (d+n) outputs; 16 x 28
// for the quadrotor: 78 % of the algorithmic flops of that kernel).  On the CUDA cores this costs
// 164 FFMA2 issue slots and 84 accumulator registers per thread; here it is one UMMA per 16 samples,
// issued by a single thread, accumulating in TMEM:
//
//     D[64 x N] (TMEM, fp32)  +=  A[64 x 16] (smem)  *  B[16 x N] (smem),     kind::f16 (bf16), MN-major
//
// A rows ("features") = [ z_1 | z_2 | dF_1 | dF_2 ],  B = the first N = 2*dq rows of the SAME smem
// array = [ z_1 | z_2 ].  Every fp32 value x is split into two bf16 pieces, x ~ x_1 - x_2' with
// x_1 = bf16_rn(x), x_2' = bf16_rn(x_1 - x)  (|x - x_1 + x_2'| <= 2^-18 |x|, round-to-nearest, so
// the residual is zero-mean and averages out over the samples; the second piece is stored negated
// because the sm_100 mixed-precision subtract FHADD.BF16 yields x_1 - x without unpacking).  D then
// holds all four partial products and their signed sum reproduces the fp32 product to ~2^-17
// relative — far inside the 1e-4 budget, and the bf16 operands halve the shared-memory traffic of a
// tf32 split (the UMMA operand reads were the bottleneck of the tf32 variant: 3 KB per 8 samples
// against 128 B/clk of smem bandwidth).
//
// MN-major canonical layout without swizzle (conventions verified on hardware by
// tools/test_umma3.cu):
//     byte address of (feature f, sample k) = (f/8)*SBO + (k/8)*LBO + (k%8)*16 + (f%8)*2
// with LBO = 128 B, SBO = (samples per tile / 8) * 128 B: a thread (lane = sample) stores 8
// consecutive features with one 16-byte STS and a warp's store covers 512 contiguous bytes.
#pragma once
#include "smooth.cuh"

#ifndef IRS_TC_NOM_BATCH
#define IRS_TC_NOM_BATCH 64
#endif
#ifndef IRS_TC_PACK_TMEM
#define IRS_TC_PACK_TMEM 1
#endif
#ifndef IRS_TC_MIN_BLOCKS
#define IRS_TC_MIN_BLOCKS 4
#endif

namespace irs {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

// 64-bit shared-memory matrix descriptor (SWIZZLE_NONE, Blackwell version bit).
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// One lane of the (converged) warp: elect.sync tells ptxas that the guarded region runs in a single
// thread, so the tcgen05 operands move to uniform registers without a vote loop per instruction.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
// Wait for the phase with the given parity to complete (try_wait suspends the thread in hardware
// for a short, implementation-defined time; the loop re-arms it).
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    }
}

// DUAL: the operand tile of a lane holds TWO sample rows ("members" 0 and 1, e.g. the + and - member of
// an antithetic pair whose projected regressors are not negatives of each other).  Possible when two
// rows fit the M = 64 operand (three_cart, bicycle, pendulum).  One UMMA pair then serves two samples:
// D [64 x 4 dq] holds the two wanted diagonal blocks (member h rows x member h columns) and two cross
// blocks that are never read.
template <class Sys, bool DUAL = false>
struct TcCfg {
    static constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    static constexpr int W = d + n;
    static constexpr int dq = (d + 7) / 8 * 8;           // regressor rows per piece (8-feature groups)
    static constexpr int nq = (n + 7) / 8 * 8;           // response rows per piece
    static constexpr int kMembers = DUAL ? 2 : 1;        // sample rows per lane and tile
    static constexpr int kN = kMembers * 2 * dq;         // UMMA N (columns of D): [z_1 | z_2] per member
    static constexpr int kRows = kMembers * (2 * dq + 2 * nq);   // used rows of A (<= 64)
    static constexpr int kM = 64;
    static constexpr int kWarps = 4;                     // self-contained warp pipelines per block
    static constexpr int kThreads = 32 * kWarps;         // lane = sample (or antithetic pair)
    static constexpr int kTile = kThreads;               // lane-units per block round
    static constexpr int kWarpTile = 32;                 // operand columns per warp tile (two K = 16 UMMAs)
    static constexpr int kLBO = 128;                     // bytes between k-groups (8 samples)
    static constexpr int kSBO = (kWarpTile / 8) * kLBO;  // bytes between 8-feature groups (512)
    static constexpr int kGroups = kM / 8;
    static constexpr int kStageBytes = kGroups * kSBO;   // 4,096 per warp tile
#if IRS_TC_PACK_TMEM
    // An M = 64 accumulator occupies lanes 0-15 of every 32-lane quarter of its TMEM columns; a second
    // one at lane offset 16 shares the columns: two warps per column range.
    static constexpr int kAccRanges = kWarps / 2;
#else
    static constexpr int kAccRanges = kWarps;                // one column range per warp
#endif
    static constexpr int kTmemCols = kAccRanges * kN < 32 ? 32 : kAccRanges * kN;
    static constexpr int NACC = gram_nacc(n, m);
    static constexpr int WIDTH = gram_width_of<Sys>();   // NACC (+ first moments, centred-capable systems)
    static constexpr int NMOM = WIDTH - NACC;
    static constexpr int RS = (W + 1) / 2 * 2;
    // Nominal points prepared per batch (one thread each).  64 for the quadrotor: batched MPC runs one
    // short item (8 rounds) per nominal point, and a per-item preparation stalls the block for ~1,400
    // cycles; 1 (per item, as measured faster) for the small systems, whose items are long.
    static constexpr int kNomBatch = d > 8 ? IRS_TC_NOM_BATCH : 1;
    static_assert(kRows <= kM, "operand rows must fit one M = 64 UMMA");
    static_assert(kN % 8 == 0 && kN >= 8 && kN <= 256, "invalid UMMA N");
    static_assert(kN % 16 == 0, "accumulator read-back uses 16-column TMEM loads");
    static_assert(kTmemCols == 32 || kTmemCols == 64 || kTmemCols == 128 || kTmemCols == 256, "TMEM allocation");
    // instruction descriptor: D fp32, A/B bf16, both MN-major, N >> 3, M >> 4
    static constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                                       ((uint32_t)(kN >> 3) << 17) | ((uint32_t)(kM >> 4) << 24);
    // feature-group index (8 rows each) of the four pieces of member h: the regressor pieces of all members
    // come first (they are the B operand = the first kN rows), then the response pieces
    __host__ __device__ static constexpr int grp_z1(int h) { return h * (2 * dq / 8); }
    __host__ __device__ static constexpr int grp_z2(int h) { return grp_z1(h) + dq / 8; }
    __host__ __device__ static constexpr int grp_f1(int h) { return kMembers * (2 * dq / 8) + h * (2 * nq / 8); }
    __host__ __device__ static constexpr int grp_f2(int h) { return grp_f1(h) + nq / 8; }
    __host__ __device__ static constexpr int row_1(int h, int j) { return j < d ? 8 * grp_z1(h) + j : 8 * grp_f1(h) + (j - d); }
    __host__ __device__ static constexpr int row_2(int h, int j) { return j < d ? 8 * grp_z2(h) + j : 8 * grp_f2(h) + (j - d); }
    // member of operand row r
    __host__ __device__ static constexpr int member_of_row(int r) {
        return r < kN ? r / (2 * dq) : (r - kN) / (2 * nq);
    }
};

// fp32 pair -> two packed bf16x2 words (low half = v0, high half = v1): first pieces p1 = bf16_rn(v)
// and NEGATED second pieces p2 = bf16_rn(p1 - v).  The residual uses the mixed-precision subtract of
// sm_100 (sub.f32.bf16 -> FHADD.BF16 with a half-register selector), so no unpacking instructions:
// 4 instructions per pair.  The sign of the second pieces is undone when the accumulator is read.
__device__ __forceinline__ void split_bf16x2(float v0, float v1, uint32_t& p1, uint32_t& p2) {
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(p1) : "f"(v1), "f"(v0));
    float n0, n1;
    asm("{\n\t.reg .b16 lo, hi;\n\tmov.b32 {lo, hi}, %2;\n\t"
        "sub.rn.f32.bf16 %0, lo, %3;\n\tsub.rn.f32.bf16 %1, hi, %4;\n\t}"
        : "=f"(n0), "=f"(n1)
        : "r"(p1), "f"(v0), "f"(v1));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(p2) : "f"(n1), "f"(n0));
}

// Persistent kernel.  A work item is one (nominal point p, sample chunk c); blocks walk the item
// list with stride gridDim.x, so the result layout (partials[p][c]) does not depend on the grid.
//
// Every warp is a self-contained pipeline: it generates 32 samples per round (lane = sample:
// Philox / replay -> perturb -> dynamics -> bf16x2 split), stages them in its OWN ring of
// shared-memory tiles, and one elected lane issues the two UMMAs (K = 16 samples each) of the tile
// into the warp's OWN accumulator in TMEM, committing them to the tile's "empty" mbarrier.  There
// is no cross-warp synchronisation inside an item: no "full" barrier, no dedicated MMA warp, no
// block barrier.  (tcgen05.mma from different threads are not ordered against each other, hence one
// accumulator per issuing warp.)  At the end of an item the block meets once: every warp reads its
// TMEM lane quarter of all four accumulators, adds them and the packed Gram block is written.
//
// MODE selects the noise source at compile time (the other paths stay out of the hot loop):
//   kTcPhilox   one Philox draw per sample (independent samples), lane = sample;
//   kTcReplay   deltas read from a.noise ([P, N, d] fp32, coalesced LDG.128), lane = sample;
//   kTcPaired   antithetic pairs (kFlagAntithetic): samples 2q and 2q + 1 are x +- z_q, lane = PAIR.
//               One Philox + Box-Muller draw serves two dynamics evaluations, and because the
//               regressors of a pair are exact negatives of each other its Gram contribution
//               collapses to ONE operand row:
//                   z z^T + (-z)(-z)^T = 2 z z^T,     z dF+^T + (-z) dF-^T = z (f(x+z) - f(x-z))^T
//               so a pair stages the row [z | f+ - f-] once (the nominal response cancels), the
//               tensor core does half the work per sample, and the regressor block is doubled when
//               the accumulator is read back (exact).  A chunk of odd length ends in a lone + member,
//               staged as [z / sqrt 2 | sqrt 2 (f+ - fbar)].  With an in-kernel projection
//               (three_cart) the projected regressors of a pair are no longer negatives: the pair
//               then shares only the noise draw and stages two rows.
enum TcMode { kTcPhilox = 0, kTcReplay = 1, kTcPaired = 2 };

// CENTERED (centred-capable systems only, gram_width_of): the regressors of the launch are relative to
// the nominal point (kFlagProjectAbsolute, or replayed absolute points with kFlagCentered) and their
// first moments [sum z' | sum dF] are appended to the packed block — per-lane fp32 sums of a few dozen
// values each, reduced by shuffles, so they carry far less rounding noise than a running sum.
// The packed pair evaluation asks for five resident blocks explicitly: left at the common cap, ptxas gives it 101
// registers (four blocks per SM); at 96 it needs no spills and one more instruction per pair.
template <class Sys, int NSTAGE, int MODE, bool CENTERED>
__global__ void __launch_bounds__(128, MODE == kTcPaired && has_step_pair<Sys>::value ? 5 : IRS_TC_MIN_BLOCKS)
    smooth_zero_order_tc_kernel(const SmoothArgs a) {
    // three_cart pairs whose regressors are projected stage both members in one tile
    constexpr bool DUAL = MODE == kTcPaired && Sys::kHasProjection;
    using C = TcCfg<Sys, DUAL>;
    constexpr int n = Sys::N, m = Sys::M, d = Sys::D;
    constexpr int kXU = (n + m + 3) / 4 * 4;             // xbar | ubar, padded to float4
    constexpr int kNom = kXU + (n + 3) / 4 * 4;          // ... | fbar, padded to float4
    constexpr int kScr = C::dq + 1;                      // padded scratch row (bank-conflict free)
    constexpr int kNomBatch = C::kNomBatch;              // nominal points prepared per batch
    constexpr int kMom = C::NMOM > 0 ? C::NMOM : 1;
    static_assert(!CENTERED || C::NMOM == d + n, "centred accumulation needs the first-moment slots");
    extern __shared__ __align__(128) unsigned char stage_mem[];   // [warp][stage][kStageBytes]
    __shared__ uint64_t mbar_empty[C::kWarps][NSTAGE];   // UMMA commit -> owning warp: tile drained
    __shared__ uint64_t mbar_done[C::kWarps];            // UMMA commit -> owning warp: accumulator complete
    __shared__ uint32_t tmem_base_s;
    // nominal points (xbar | ubar | f(xbar, ubar), fp32) of this block's next kNomBatch items, prepared
    // kNomBatch at a time by one thread each: the loads and the scalar dynamics at the nominal then
    // cost one latency per batch instead of one per item
    __shared__ __align__(16) float nom_tab[kNomBatch][kNom];
    __shared__ double pos64_tab[kNomBatch][4];           // leading coordinates in fp64 (projection)
    __shared__ double nom64_s[n + m];                    // fp64 nominal of the current item (kNomBatch == 1)
    __shared__ float scratch[C::kRows * kScr];           // s_r[i] = D[r][z_1 col i] - D[r][z_2 col i] of r's member
    __shared__ uint16_t idx_s[C::NACC];                  // packed output e -> (i << 8) | j
    __shared__ float mom_s[C::kWarps][kMom];             // per-warp first moments of the item

    const int tid = threadIdx.x, lane = tid & 31;
    // broadcast from lane 0 so that the compiler knows the warp index is warp-uniform: ring addresses,
    // descriptors and barrier addresses then live in uniform registers (fewer R2UR around the UMMAs)
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const long long num_items = (long long)a.P * a.C;

    if (tid == 0) {
#pragma unroll
        for (int w = 0; w < C::kWarps; ++w) {
#pragma unroll
            for (int s = 0; s < NSTAGE; ++s) mbar_init(&mbar_empty[w][s], 1);
            mbar_init(&mbar_done[w], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    for (int e = tid; e < C::NACC; e += C::kThreads) {
        int i = 0;
        while (i + 1 < d && gram_row_offset(i + 1, C::W) <= e) ++i;
        idx_s[e] = (uint16_t)((i << 8) | (i + (e - gram_row_offset(i, C::W))));
    }
    if constexpr (DUAL) {
        // a launch that stages one row per lane (no projection) never writes the second member's rows
        for (int e = tid; e < NSTAGE * C::kWarps * C::kStageBytes / 16; e += C::kThreads)
            reinterpret_cast<uint4*>(stage_mem)[e] = make_uint4(0u, 0u, 0u, 0u);
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"(C::kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    const Sys sys(a.prm);
    // The point (xb | ub) the samples are perturbed around and the response fb every sample's f is measured
    // against.  Ordinarily the fp32 nominal and the scalar dynamics there (…zero_order.py:52).  CENTERED
    // (regressors are absolute points xbar + z', so the state of a sample is 2 xbar + z'): the doubled
    // nominal in the system's centred frame (systems.cuh: centred_frame) and the SAMPLE dynamics there, so
    // that the accumulated responses are O(sigma) like the regressors — f(2 xbar + z') - f(xbar) itself is
    // ~ |xbar|, and a fp32 sum of it, multiplied by the shift |xbar| when the fit is un-centred, would cost
    // |xbar|^2 in accuracy.  The finalize adds f_batch(2 xbar, 2 ubar) - f(xbar, ubar) back in fp64.
    auto nominal_point = [&](int p, int slot, float (&xb)[n], float (&ub)[m], float (&fb)[n]) {
        double xd[n], ud[m];
#pragma unroll
        for (int q = 0; q < n; ++q) {
            xd[q] = a.x_nom[(long long)p * n + q];
            if (q < 4) pos64_tab[slot][q] = xd[q];
        }
#pragma unroll
        for (int q = 0; q < m; ++q) ud[q] = a.u_nom[(long long)p * m + q];
        if constexpr (CENTERED) {
            centred_frame<Sys>(xd, ud, xb, ub);
            if (a.flags & kFlagSamplesBatchVariant) sys.template step<true>(xb, ub, fb);
            else sys.template step<false>(xb, ub, fb);
        } else {
#pragma unroll
            for (int q = 0; q < n; ++q) xb[q] = (float)xd[q];
#pragma unroll
            for (int q = 0; q < m; ++q) ub[q] = (float)ud[q];
            sys.template step<false>(xb, ub, fb);
        }
    };
    // nominal points of the items first, first + gridDim.x, ... -> nom_tab, one thread each (all threads
    // call it; the caller's barriers order it against the readers)
    auto prepare_nominals = [&](long long first) {
        if (tid < kNomBatch) {
            const long long it2 = first + (long long)tid * gridDim.x;
            if (it2 < num_items) {
                float xb[n], ub[m], fb[n];
                nominal_point((int)(it2 / a.C), tid, xb, ub, fb);
                float* row = nom_tab[tid];
#pragma unroll
                for (int q = 0; q < n; ++q) row[q] = xb[q];
#pragma unroll
                for (int q = 0; q < m; ++q) row[n + q] = ub[q];
#pragma unroll
                for (int q = n + m; q < kXU; ++q) row[q] = 0.f;
#pragma unroll
                for (int q = 0; q < n; ++q) row[kXU + q] = fb[q];
            }
        }
    };
    // kNomBatch == 1: the nominal point of one item, cooperatively (the threads fetch the coordinates in
    // parallel, thread 0 evaluates the reference response; two block barriers inside)
    auto load_nominal = [&](long long item) {
        const int p = (int)(item / a.C);
        float* nom_s = nom_tab[0];
        if (tid < n) nom64_s[tid] = a.x_nom[(long long)p * n + tid];
        else if (tid < n + m) nom64_s[tid] = a.u_nom[(long long)p * m + (tid - n)];
        __syncthreads();
        if (tid < 4 && tid < n) pos64_tab[0][tid] = nom64_s[tid];
        if (tid == 0) {
            float xb[n], ub[m], fb[n];
            if constexpr (CENTERED) {
                double xd[n], ud[m];
#pragma unroll
                for (int q = 0; q < n; ++q) xd[q] = nom64_s[q];
#pragma unroll
                for (int q = 0; q < m; ++q) ud[q] = nom64_s[n + q];
                centred_frame<Sys>(xd, ud, xb, ub);
                if (a.flags & kFlagSamplesBatchVariant) sys.template step<true>(xb, ub, fb);
                else sys.template step<false>(xb, ub, fb);
            } else {
#pragma unroll
                for (int q = 0; q < n; ++q) xb[q] = (float)nom64_s[q];
#pragma unroll
                for (int q = 0; q < m; ++q) ub[q] = (float)nom64_s[n + q];
                sys.template step<false>(xb, ub, fb);   // scalar dynamics at the nominal (…zero_order.py:52)
            }
#pragma unroll
            for (int q = 0; q < n; ++q) nom_s[q] = xb[q];
#pragma unroll
            for (int q = 0; q < m; ++q) nom_s[n + q] = ub[q];
#pragma unroll
            for (int q = 0; q < n; ++q) nom_s[kXU + q] = fb[q];
        }
        __syncthreads();
    };
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem_base = tmem_base_s;
#if IRS_TC_PACK_TMEM
    const uint32_t tmem_acc = tmem_base + ((uint32_t)(16 * (warp & 1)) << 16) + (uint32_t)((warp >> 1) * C::kN);
#else
    const uint32_t tmem_acc = tmem_base + (uint32_t)(warp * C::kN);      // this warp's accumulator
#endif

    [[maybe_unused]] const bool batch = (a.flags & kFlagSamplesBatchVariant) != 0;
    // this warp's tile ring; byte offset of this lane's sample inside a tile (feature group 0)
    unsigned char* my_ring = stage_mem + (size_t)warp * NSTAGE * C::kStageBytes;
    const uint32_t ring_u32 = smem_u32(my_ring);
    const uint32_t my_off = (uint32_t)(lane >> 3) * C::kLBO + (uint32_t)(lane & 7) * 16;

    // Issue the UMMAs of a staged tile (all lanes call it; one lane issues).
    auto issue_tile = [&](int stage, bool first, bool last) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> async proxy
        __syncwarp();
        if (elect_one()) {
            const uint64_t desc0 = umma_smem_desc(ring_u32 + stage * C::kStageBytes, C::kLBO, C::kSBO);
#pragma unroll
            for (int kb = 0; kb < C::kWarpTile / 16; ++kb) {   // one UMMA = K 16 = two k-groups of 8 samples
                const uint64_t desc = desc0 + (uint64_t)((kb * 2 * C::kLBO) >> 4);
                const uint32_t acc = (!first || kb > 0) ? 1u : 0u;   // first UMMA of an item overwrites
                asm volatile(
                    "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                    "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_acc),
                    "l"(desc), "l"(desc), "r"(C::kIdesc), "r"(acc)
                    : "memory");
            }
            // frees the tile once these UMMAs have read it (commit implies fence::before_thread_sync)
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                             smem_u32(&mbar_empty[warp][stage]))
                         : "memory");
            if (last)
                asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                                 smem_u32(&mbar_done[warp]))
                             : "memory");
        }
        __syncwarp();
    };

    int round = 0;      // running tile counter of this warp (tile ring position)
    int it = 0;         // running item counter of this block
    for (long long item = blockIdx.x; item < num_items; item += gridDim.x, ++it) {
        const int p = (int)(item / a.C);
        const int c = (int)(item % a.C);
        const long long s_begin = (long long)c * a.S;
        const long long s_end = s_begin + a.S < a.N ? s_begin + a.S : a.N;
        const int slot = kNomBatch == 1 ? 0 : it % kNomBatch;
        if constexpr (kNomBatch == 1) {
            load_nominal(item);
        } else {
            if (slot == 0) {
                if (it > 0) __syncthreads();      // every warp is done with the previous batch of nominal points
                prepare_nominals(item);
                __syncthreads();
            }
        }
        const float4* nom4 = reinterpret_cast<const float4*>(nom_tab[slot]);
        const double* pos64_s = pos64_tab[slot];
        float mom[kMom];                                      // first moments of this lane's rows (CENTERED)
#pragma unroll
        for (int q = 0; q < kMom; ++q) mom[q] = 0.f;
        // the nominal point stays in shared memory (broadcast LDS.128 instead of 28 registers: measured
        // faster than the register copy)
        auto load_xu = [&](float (&xu)[kXU]) {
#pragma unroll
            for (int q = 0; q < kXU / 4; ++q) {
                const float4 v = nom4[q];
                xu[4 * q] = v.x;  xu[4 * q + 1] = v.y;  xu[4 * q + 2] = v.z;  xu[4 * q + 3] = v.w;
            }
        };
        // xu = nominal point + w
        auto perturb = [&](float (&xu)[kXU], const float (&w)[C::RS]) {
#pragma unroll
            for (int q = 0; q < d; ++q) xu[q] += w[q];
        };
        auto dynamics = [&](const float (&xu)[kXU], float (&f)[n]) {
            if constexpr (Sys::kHasProjection) {    // only three_cart distinguishes batch / scalar
                if (batch) sys.template step<true>(xu, xu + n, f);
                else sys.template step<false>(xu, xu + n, f);
            } else {
                sys.template step<false>(xu, xu + n, f);
            }
        };
        // w = [z | f(x̄ + z) - f(x̄ - z)] of an antithetic pair, both members evaluated at once in the two halves
        // of packed FP32 registers: half the issue slots of two scalar evaluations, the same bits.  z arrives in
        // both halves of a register pair, so (x̄ + z, x̄ - z) is one FADD2 whose operand negates the high half.
        auto pair_row = [&](unsigned long long pair, float (&w)[C::RS]) {
            if constexpr (has_step_pair<Sys>::value) {
                float2 xu2[d], f2[n];
#pragma unroll
                for (int j = 0; j < (d + 3) / 4; ++j) {     // block by block: a block's z pairs die at once
                    float2 zz[4];
                    philox_normals_x2<Sys>(a, p, pair, j, zz);
                    const float4 v = nom4[j];
                    const float xb[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (4 * j + k < d) {
                            w[4 * j + k] = zz[k].x;
                            xu2[4 * j + k] = Lanes<float2>::add(Lanes<float2>::splat(xb[k]), make_float2(zz[k].x, -zz[k].y));
                        }
                    }
                }
                sys.step_pair(xu2, xu2 + n, f2);
#pragma unroll
                for (int q = 0; q < n; ++q) w[d + q] = f2[q].x - f2[q].y;
            }
        };
        // w[d ..] = scale (f - fbar)
        auto minus_nominal_response = [&](const float (&f)[n], float (&w)[C::RS], float scale) {
#pragma unroll
            for (int q = 0; q < (n + 3) / 4; ++q) {
                const float4 v = nom4[kXU / 4 + q];
                const float fb[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (4 * q + k < n) w[d + 4 * q + k] = scale * (f[4 * q + k] - fb[k]);
            }
        };
        // one ordinary sample row: deltas w[0 .. d) -> projected / perturbed / evaluated -> w = [z | dF]
        auto finish_row = [&](float (&w)[C::RS]) {
            float xu[kXU], f[n];
            load_xu(xu);
            project_deltas<Sys, C::RS>(a, p, pos64_s, w);
            if constexpr (CENTERED && MODE == kTcReplay) {
                // replayed absolute points -> relative to the nominal (the state below is frame + w)
                if (!(a.flags & kFlagProjectAbsolute)) center_replayed<Sys, C::RS>(a, p, w);
            }
            perturb(xu, w);
            dynamics(xu, f);
            minus_nominal_response(f, w, 1.f);
            if constexpr (CENTERED) {
#pragma unroll
                for (int q = 0; q < d + n; ++q) mom[q] += w[q];
            }
        };
        auto zero_row = [&](float (&w)[C::RS]) {
#pragma unroll
            for (int q = 0; q < C::RS; ++q) w[q] = 0.f;      // ragged tail: contributes nothing
        };
        // The tile must have been drained by the UMMAs that last read it (call before its first store).
        auto wait_tile = [&]() {
            const int stage = round % NSTAGE;
            if (round >= NSTAGE) mbar_wait(&mbar_empty[warp][stage], (uint32_t)((round / NSTAGE - 1) & 1));
        };
        // One operand row of this lane -> member h of the warp's current tile (bf16x2 split, MN-major).
        auto stage_row = [&](const float (&w)[C::RS], auto member_tag) {
            constexpr int h = decltype(member_tag)::value;
            unsigned char* sm = my_ring + (round % NSTAGE) * C::kStageBytes + my_off;
            // regressors: dq/8 groups of 8 features, first and second bf16 pieces
#pragma unroll
            for (int g = 0; g < C::dq / 8; ++g) {
                uint32_t p1[4], p2[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c0 = 8 * g + 2 * q, c1 = c0 + 1;
                    // padding rows are zero at compile time (inline asm is not constant-folded)
                    if (c0 < d) split_bf16x2(w[c0], c1 < d ? w[c1] : 0.f, p1[q], p2[q]);
                    else p1[q] = p2[q] = 0u;
                }
                *reinterpret_cast<uint4*>(sm + (C::grp_z1(h) + g) * C::kSBO) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
                *reinterpret_cast<uint4*>(sm + (C::grp_z2(h) + g) * C::kSBO) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
            }
            // responses
#pragma unroll
            for (int g = 0; g < C::nq / 8; ++g) {
                uint32_t p1[4], p2[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int c0 = 8 * g + 2 * q, c1 = c0 + 1;
                    if (c0 < n) split_bf16x2(w[d + c0], c1 < n ? w[d + c1] : 0.f, p1[q], p2[q]);
                    else p1[q] = p2[q] = 0u;
                }
                *reinterpret_cast<uint4*>(sm + (C::grp_f1(h) + g) * C::kSBO) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
                *reinterpret_cast<uint4*>(sm + (C::grp_f2(h) + g) * C::kSBO) = make_uint4(p2[0], p2[1], p2[2], p2[3]);
            }
        };
        auto issue = [&](bool first, bool last) {
            issue_tile(round % NSTAGE, first, last);
            ++round;
        };
        using Member0 = std::integral_constant<int, 0>;
        using Member1 = std::integral_constant<int, DUAL ? 1 : 0>;
        const long long len = s_end - s_begin;                // samples of this chunk
        // pairs share a noise draw only (two operand rows per pair) when the regressors are projected
        [[maybe_unused]] const bool pair_rows =
            Sys::kHasProjection && (a.flags & (kFlagProjectAbsolute | kFlagProjectDelta)) != 0;
        const long long units = MODE == kTcPaired ? (len + 1) / 2 : len;      // lanes of work: pairs or samples
        const int rounds = (int)((units + C::kTile - 1) / C::kTile);
        // One round = one lane-unit per thread (a sample, or an antithetic pair).  CHECK = false is the
        // hot path (every lane owns a full unit); only the last round of a chunk whose length is not a
        // multiple of the tile takes the CHECK = true path, where missing samples stage zeros.
        auto do_round = [&](auto check_tag, int r) {
            constexpr bool CHECK = decltype(check_tag)::value;
            const long long lu = (long long)r * C::kTile + tid;       // this lane's unit inside the chunk
            const bool first = r == 0, last = r == rounds - 1;
            float w[C::RS];
            if constexpr (C::RS > C::W) w[C::RS - 1] = 0.f;
            if constexpr (MODE != kTcPaired) {
                if (!CHECK || lu < len) {
                    draw_deltas<Sys, C::RS, MODE == kTcReplay ? 1 : 0>(a, p, s_begin + lu, w);
                    finish_row(w);
                } else {
                    zero_row(w);
                }
                wait_tile();
                stage_row(w, Member0{});
                issue(first, last);
            } else {
                const bool have_plus = !CHECK || 2 * lu < len;
                const bool have_minus = !CHECK || 2 * lu + 1 < len;
                // the pair's draw: counter word 0 = global pair index (a.i0 and s_begin are even)
                const unsigned long long pair = ((a.i0 + (unsigned long long)s_begin) >> 1) + (unsigned long long)lu;
                bool two_rows = false;
                if constexpr (DUAL) two_rows = pair_rows;
                if (!two_rows) {
                    if (have_plus) {
                        if (has_step_pair<Sys>::value && have_minus) {
                            pair_row(pair, w);
                        } else {
                            philox_normals<Sys, C::RS>(a, p, pair, w);
                            float xu[kXU], fp[n];
                            load_xu(xu);
#pragma unroll
                            for (int q = 0; q < d; ++q) xu[q] += w[q];
                            dynamics(xu, fp);
                            if (have_minus) {
                                float fm[n];
                                load_xu(xu);
#pragma unroll
                                for (int q = 0; q < d; ++q) xu[q] -= w[q];
                                dynamics(xu, fm);
#pragma unroll
                                for (int q = 0; q < n; ++q) w[d + q] = fp[q] - fm[q];
                            } else {
                                // lone + member at the end of an odd chunk: [z / sqrt 2 | sqrt 2 (f+ - fbar)]
                                minus_nominal_response(fp, w, 1.41421356237309505f);
#pragma unroll
                                for (int q = 0; q < d; ++q) w[q] *= 0.70710678118654752f;
                            }
                        }
                    } else {
                        zero_row(w);
                    }
                    wait_tile();
                    stage_row(w, Member0{});
                    issue(first, last);
                } else {
                    if constexpr (DUAL) {
                        // both members of the pair in ONE tile: + member rows, then - member rows
                        float z[d];
                        if (have_plus) {
                            philox_normals<Sys, C::RS>(a, p, pair, w);
#pragma unroll
                            for (int q = 0; q < d; ++q) z[q] = w[q];
                            finish_row(w);
                        } else {
#pragma unroll
                            for (int q = 0; q < d; ++q) z[q] = 0.f;
                            zero_row(w);
                        }
                        wait_tile();
                        stage_row(w, Member0{});
                        if (have_minus) {
#pragma unroll
                            for (int q = 0; q < d; ++q) w[q] = -z[q];
                            finish_row(w);
                        } else {
                            zero_row(w);
                        }
                        stage_row(w, Member1{});
                        issue(first, last);
                    }
                }
            }
        };
        const int full_rounds = (int)((MODE == kTcPaired ? len / 2 : len) / C::kTile);
        for (int r = 0; r < full_rounds; ++r) do_round(std::false_type{}, r);
        if (full_rounds < rounds) do_round(std::true_type{}, full_rounds);
        if constexpr (CENTERED) {
            // first moments of the item: lanes -> warp (shuffles) -> block (shared memory, fixed order below)
#pragma unroll
            for (int q = 0; q < d + n; ++q) {
                const float v = warp_sum(mom[q]);
                if (lane == 0) mom_s[warp][q] = v;
            }
        }
        // ---- item finished: wait for this warp's UMMAs, meet the other warps, read all four
        //      accumulators back.  Row r of D lives in TMEM lane (r % 16) + 32 * (r / 16) (M = 64
        //      layout): lanes 0-15 of warp w hold rows 16 w .. 16 w + 15 of every accumulator (and
        //      lanes 16-31 the same rows of the accumulators packed at lane offset 16). ----
        mbar_wait(&mbar_done[warp], (uint32_t)(it & 1));
        asm volatile("tcgen05.fence::before_thread_sync;");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;");
        {
            float sum[C::kN];
#pragma unroll
            for (int q = 0; q < C::kN; ++q) sum[q] = 0.f;
            const uint32_t taddr = tmem_base + ((uint32_t)(32 * warp) << 16);
#pragma unroll
            for (int wa = 0; wa < C::kAccRanges; ++wa) {
                uint32_t v[C::kN];
#pragma unroll
                for (int c0 = 0; c0 < C::kN; c0 += 16) {
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                        : "=r"(v[c0 + 0]), "=r"(v[c0 + 1]), "=r"(v[c0 + 2]), "=r"(v[c0 + 3]), "=r"(v[c0 + 4]),
                          "=r"(v[c0 + 5]), "=r"(v[c0 + 6]), "=r"(v[c0 + 7]), "=r"(v[c0 + 8]), "=r"(v[c0 + 9]),
                          "=r"(v[c0 + 10]), "=r"(v[c0 + 11]), "=r"(v[c0 + 12]), "=r"(v[c0 + 13]), "=r"(v[c0 + 14]),
                          "=r"(v[c0 + 15])
                        : "r"(taddr + (uint32_t)(wa * C::kN + c0)));
                }
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
                for (int q = 0; q < C::kN; ++q) sum[q] += __uint_as_float(v[q]);    // fixed warp order
            }
#if IRS_TC_PACK_TMEM
            // lanes 16-31 of the quarter hold the same rows of the accumulators at lane offset 16
#pragma unroll
            for (int q = 0; q < C::kN; ++q) sum[q] += __shfl_down_sync(0xffffffffu, sum[q], 16);
#endif
            const int row = 16 * warp + lane;
            if (lane < 16 && row < C::kRows) {
                // columns of the row's OWN member: z_1 piece minus z_2 piece (the z_2 columns are negated)
                const bool second = C::member_of_row(row) == 1;
#pragma unroll
                for (int i = 0; i < C::dq; ++i) {
                    float v = sum[i] - sum[C::dq + i];
                    if constexpr (DUAL) {
                        const float v1 = sum[2 * C::dq + i] - sum[3 * C::dq + i];
                        v = second ? v1 : v;
                    }
                    scratch[row * kScr + i] = v;
                }
            }
        }
        asm volatile("tcgen05.fence::before_thread_sync;");
        __syncthreads();      // scratch complete; every accumulator read back (next item may overwrite)
        asm volatile("tcgen05.fence::after_thread_sync;");
        // G[i][j] = sum_k z_i w_j = sum over the two pieces of w_j of s_row[i] (second-piece rows negated),
        // summed over the members of the tile
        float* out = a.partials + item * C::WIDTH;
        // paired rows: the regressor block of a pair is 2 z z^T (exact doubling)
        const float zz_scale = (MODE == kTcPaired && !pair_rows) ? 2.f : 1.f;
        for (int e = tid; e < C::NACC; e += C::kThreads) {
            const int ij = idx_s[e];
            const int i = ij >> 8, j = ij & 0xff;
            float v = scratch[C::row_1(0, j) * kScr + i] - scratch[C::row_2(0, j) * kScr + i];
            if constexpr (DUAL) v += scratch[C::row_1(1, j) * kScr + i] - scratch[C::row_2(1, j) * kScr + i];
            out[e] = j < d ? zz_scale * v : v;
        }
        if constexpr (C::NMOM > 0) {
            if (tid < C::NMOM) {
                float v = 0.f;
                if constexpr (CENTERED) v = (mom_s[0][tid] + mom_s[1][tid]) + (mom_s[2][tid] + mom_s[3][tid]);
                out[C::NACC + tid] = v;
            }
        }
        // (the next item's barriers order these scratch / mom_s reads before the next writes)
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(C::kTmemCols));
}

}  // namespace irs
