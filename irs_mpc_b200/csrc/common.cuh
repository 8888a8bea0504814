// Shared device helpers for the iRS-MPC sm_100a kernels: error plumbing, Philox4x32,
// Box-Muller, packed-FP32 FMA (FFMA2), scalar-type math wrappers.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace irs {

// ---------------------------------------------------------------------------------------------
// Error plumbing (C-ABI returns int status; message retrievable through irs_last_error()).
// ---------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define IRS_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            irs::set_error(__VA_ARGS__);  \
            return 1;                     \
        }                                 \
    } while (0)

// System parameters travel by value into the kernels (<= 10 doubles).  `f` mirrors `v` in fp32
// followed by the derived loop invariants of the system (filled on the host in double precision,
// load_params in api.cu), so that the fp32 sample kernels read them as constant-bank operands
// instead of converting doubles (F2F runs on the XU pipe, the busiest one in the sample loop).
struct SysParams {
    double v[10];
    float f[20];
    // learned dynamics (systems.cuh: Mlp): device blob of the registered network, hidden widths
    const float* mlp;
    const unsigned short* mlp_w2;      // hidden layer as tensor-core operand: bf16 pieces [hi | lo] (smooth_mlp.cuh)
    int h1, h2;
};

// ---------------------------------------------------------------------------------------------
// Scalar math wrappers.  float: MUFU-backed fast intrinsics (the sample path is throughput
// bound and the least-squares fit averages their ~1e-7 absolute error away); double: libdevice.
// ---------------------------------------------------------------------------------------------
template <typename R>
struct Math;

template <>
struct Math<float> {
    static __device__ __forceinline__ void sincos(float a, float& s, float& c) {
        __sincosf(a, &s, &c);
    }
    static __device__ __forceinline__ float rcp(float a) {
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a));      // one MUFU.RCP, no slow path
        return r;
    }
    static __device__ __forceinline__ float div(float a, float b) { return __fdividef(a, b); }
};

template <>
struct Math<double> {
    static __device__ __forceinline__ void sincos(double a, double& s, double& c) {
        ::sincos(a, &s, &c);
    }
    static __device__ __forceinline__ double rcp(double a) { return 1.0 / a; }
    static __device__ __forceinline__ double div(double a, double b) { return a / b; }
};

// ---------------------------------------------------------------------------------------------
// Philox4x32 (Salmon et al., SC'11).  Spec of the counter layout: oracle/philox_ref.py.
// The sample stream uses kPhiloxRounds = 7 rounds: the smallest round count of Philox4x32 that
// the paper reports as Crush-resistant (10 is its default safety margin).  On sm_100a the two
// 32x32->64 multiplies per round issue at a quarter of the FP32 rate (measured: 32
// IMAD.WIDE/clk/SM vs 128 FFMA/clk/SM), so the rounds are the single largest item of the
// sample-generation cost.  The round function itself is pinned on the Random123 10-round
// known-answer vectors (tests/test_oracle_philox.py).
// ---------------------------------------------------------------------------------------------
constexpr int kPhiloxRounds = 7;
constexpr uint32_t kPhiloxM0 = 0xD2511F53u;
constexpr uint32_t kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u;
constexpr uint32_t kPhiloxW1 = 0xBB67AE85u;

template <int ROUNDS = kPhiloxRounds>
__device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                           uint32_t k0, uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < ROUNDS; ++r) {
        const uint32_t hi0 = __umulhi(kPhiloxM0, c0);
        const uint32_t lo0 = kPhiloxM0 * c0;
        const uint32_t hi1 = __umulhi(kPhiloxM1, c2);
        const uint32_t lo1 = kPhiloxM1 * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += kPhiloxW0;
        k1 += kPhiloxW1;
    }
    out[0] = c0;
    out[1] = c1;
    out[2] = c2;
    out[3] = c3;
}

// float in [1,2) from the top 23 bits of w (exact).
__device__ __forceinline__ float unit_float(uint32_t w) {
    return __uint_as_float((w >> 9) | 0x3f800000u);
}

// Box-Muller on two 32-bit words, returned UNSCALED:  (g0, g1) = sqrt(-log2 u) * (cos, sin)(2 pi f)
// with u = 2 - unit_float(wa) in (0,1] and f = unit_float(wb) in [1,2).  The standard normals of
// the spec (oracle/philox_ref.py: angle 2 pi (f - 1.5), radius sqrt(-2 ln u)) are
//     e = -sqrt(2 ln 2) * g        (cos/sin(x - 3 pi) = -cos/sin(x))
// so callers fold kBoxMullerScale into sigma once instead of spending FMULs per sample.
constexpr float kBoxMullerScale = -1.1774100225154747f;     // -sqrt(2 ln 2)

__device__ __forceinline__ void box_muller_raw(uint32_t wa, uint32_t wb, float& g0, float& g1) {
    const float u = 2.0f - unit_float(wa);                      // (0, 1]
    float l2, r;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u));      // MUFU.LG2 (u >= 2^-23: never denormal)
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(-l2));    // MUFU.SQRT
    float s, c;
    __sincosf(unit_float(wb) * 6.283185307179586f, &s, &c);     // argument in [2 pi, 4 pi)
    g0 = r * c;
    g1 = r * s;
}

// ---------------------------------------------------------------------------------------------
// Packed FP32 FMA (Blackwell FFMA2): d = a * b + c on two lanes, one issue slot.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    uint64_t ua, ub, uc, ud;
    ua = *reinterpret_cast<uint64_t*>(&a);
    ub = *reinterpret_cast<uint64_t*>(&b);
    uc = *reinterpret_cast<uint64_t*>(&c);
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(ud) : "l"(ua), "l"(ub), "l"(uc));
    return *reinterpret_cast<float2*>(&ud);
}

// ---------------------------------------------------------------------------------------------
// fp32 arithmetic with every rounding explicit, on one value (float) or on both halves of a float2 in
// one instruction (FADD2 / FMUL2 / FFMA2).  Nothing is contracted or re-associated, so one source
// rounds identically on either type, lane by lane.  ptxas folds a splat into the .F32 (broadcast)
// operand selector and a negated pair into the operand's sign modifier: neither costs an instruction.
// ---------------------------------------------------------------------------------------------
template <typename V>
struct Lanes;

template <>
struct Lanes<float> {
    static __device__ __forceinline__ float splat(float a) { return a; }
    static __device__ __forceinline__ float neg(float a) { return -a; }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float fma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
    static __device__ __forceinline__ float rcp(float a) { return Math<float>::rcp(a); }
};

#define IRS_F32X2_BINARY(OP)                                                                            \
    float2 d;                                                                                           \
    asm("{\n\t.reg .b64 a, b, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\t" OP             \
        ".rn.f32x2 d, a, b;\n\tmov.b64 {%0, %1}, d;\n\t}"                                               \
        : "=f"(d.x), "=f"(d.y)                                                                          \
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                                      \
    return d;

template <>
struct Lanes<float2> {
    static __device__ __forceinline__ float2 splat(float a) { return make_float2(a, a); }
    static __device__ __forceinline__ float2 neg(float2 a) { return make_float2(-a.x, -a.y); }
    static __device__ __forceinline__ float2 add(float2 a, float2 b) { IRS_F32X2_BINARY("add") }
    static __device__ __forceinline__ float2 sub(float2 a, float2 b) { IRS_F32X2_BINARY("sub") }
    static __device__ __forceinline__ float2 mul(float2 a, float2 b) { IRS_F32X2_BINARY("mul") }
    static __device__ __forceinline__ float2 fma(float2 a, float2 b, float2 c) {
        float2 d;
        asm("{\n\t.reg .b64 a, b, c, d;\n\tmov.b64 a, {%2, %3};\n\tmov.b64 b, {%4, %5};\n\tmov.b64 c, {%6, %7};\n\t"
            "fma.rn.f32x2 d, a, b, c;\n\tmov.b64 {%0, %1}, d;\n\t}"
            : "=f"(d.x), "=f"(d.y)
            : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
        return d;
    }
    static __device__ __forceinline__ float2 rcp(float2 a) { return make_float2(Math<float>::rcp(a.x), Math<float>::rcp(a.y)); }
};
#undef IRS_F32X2_BINARY

// box_muller_raw on the word pairs (wa0, wb0) -> e01 and (wa1, wb1) -> e23 with the float arithmetic of the
// two packed: the bits of two box_muller_raw calls.
__device__ __forceinline__ void box_muller_raw_x2(uint32_t wa0, uint32_t wb0, uint32_t wa1, uint32_t wb1,
                                                  float2& e01, float2& e23) {
    using L = Lanes<float2>;
    const float2 u = L::sub(L::splat(2.0f), make_float2(unit_float(wa0), unit_float(wa1)));
    const float2 ang = L::mul(make_float2(unit_float(wb0), unit_float(wb1)), L::splat(6.283185307179586f));
    float l2a, l2b, ra, rb;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2a) : "f"(u.x));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2b) : "f"(u.y));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(ra) : "f"(-l2a));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rb) : "f"(-l2b));
    float sa, ca, sb, cb;
    __sincosf(ang.x, &sa, &ca);
    __sincosf(ang.y, &sb, &cb);
    e01 = L::mul(L::splat(ra), make_float2(ca, sa));
    e23 = L::mul(L::splat(rb), make_float2(cb, sb));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace irs
