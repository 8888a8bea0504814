// Forward-mode dual numbers for user-written dynamics (irs_mpc_b200/user_system.py, autodiff=True).
//
// Dual<R, K> is a value of type R (float or double) and K tangent lanes: d(value) / d(seed column k).  A user
// library built with autodiff evaluates its step body over Dual<R, K> in P passes of K columns each and reads the
// Jacobian off the tangents (UserSystem::jac_var, generated).  Only the translation unit of such a library
// includes this header (IRS_USER_AUTODIFF); the main library and the other user libraries never see it.
//
// Tangent storage: float keeps its tangents as float2 pairs (K rounded up to even) and does every tangent
// multiply and add with the packed .f32x2 instructions of Lanes<float2> (FMUL2 / FADD2 / FFMA2, common.cuh):
// the tangent work is K-wide elementwise multiply-adds, two lanes per issue slot.  double keeps K scalars.
//
// Dual and its free functions live in irs::ad, where only argument-dependent lookup finds them: an overload
// such as sqrt(Dual) declared in namespace irs would stop the unqualified lookup of sqrt(float) in a plain body
// there.  There is no conversion from Dual back to R, so a body that drops the derivative (`float t = x[0];`,
// `(int)x[0]`) does not compile.
//
// Semantics at kinks: comparisons and branches follow the values; fabs at 0 takes the + branch; fmin / fmax
// take the tangent of the argument they select, the first one on a tie; sqrt at 0 has the infinite derivative
// that math gives (a lane whose tangent is 0 then reads NaN).
#pragma once
#include <type_traits>

#include "common.cuh"

namespace irs {
namespace ad {

// tangent storage and arithmetic of one scalar type: lanes of type T, `count(K)` of them for K tangents
template <typename R>
struct Tan;

template <>
struct Tan<float> {
    using T = float2;
    using L = Lanes<float2>;
    static constexpr int count(int K) { return (K + 1) / 2; }
    static __device__ __forceinline__ T zero() { return make_float2(0.f, 0.f); }
    static __device__ __forceinline__ T splat(float a) { return L::splat(a); }
    static __device__ __forceinline__ T neg(T a) { return L::neg(a); }
    static __device__ __forceinline__ T add(T a, T b) { return L::add(a, b); }
    static __device__ __forceinline__ T sub(T a, T b) { return L::sub(a, b); }
    static __device__ __forceinline__ T mul(T a, T b) { return L::mul(a, b); }
    static __device__ __forceinline__ T fma(T a, T b, T c) { return L::fma(a, b, c); }
    static __device__ __forceinline__ float get(const T* t, int k) { return (k & 1) ? t[k >> 1].y : t[k >> 1].x; }
    static __device__ __forceinline__ void set(T* t, int k, float v) {
        if (k & 1) t[k >> 1].y = v;
        else t[k >> 1].x = v;
    }
};

template <>
struct Tan<double> {
    using T = double;
    static constexpr int count(int K) { return K; }
    static __device__ __forceinline__ T zero() { return 0.0; }
    static __device__ __forceinline__ T splat(double a) { return a; }
    static __device__ __forceinline__ T neg(T a) { return -a; }
    static __device__ __forceinline__ T add(T a, T b) { return a + b; }
    static __device__ __forceinline__ T sub(T a, T b) { return a - b; }
    static __device__ __forceinline__ T mul(T a, T b) { return a * b; }
    static __device__ __forceinline__ T fma(T a, T b, T c) { return ::fma(a, b, c); }
    static __device__ __forceinline__ double get(const T* t, int k) { return t[k]; }
    static __device__ __forceinline__ void set(T* t, int k, double v) { t[k] = v; }
};

template <typename A>
using if_arith = std::enable_if_t<std::is_arithmetic<A>::value, int>;

template <typename R, int K>
struct Dual {
    static_assert(std::is_same<R, float>::value || std::is_same<R, double>::value, "Dual<float or double, K>");
    static_assert(K >= 1, "at least one tangent");
    using Ops = Tan<R>;
    using T = typename Ops::T;
    static constexpr int L = Ops::count(K);
    R v;
    T t[L];

    Dual() = default;
    // a constant: zero tangent
    template <typename A, if_arith<A> = 0>
    __device__ __forceinline__ Dual(A a) : v(R(a)) {
#pragma unroll
        for (int i = 0; i < L; ++i) t[i] = Ops::zero();
    }
    // the value of column `col` of a pass: unit tangent in lane col (none when col is outside [0, K))
    static __device__ __forceinline__ Dual seed(R a, int col) {
        Dual r(a);
        if (col >= 0 && col < K) Ops::set(r.t, col, R(1));
        return r;
    }
    __device__ __forceinline__ R tangent(int k) const { return Ops::get(t, k); }
    // value f(v) with derivative df: tangents df * t
    __device__ __forceinline__ Dual chain(R fv, R df) const {
        Dual r;
        r.v = fv;
        const T s = Ops::splat(df);
#pragma unroll
        for (int i = 0; i < L; ++i) r.t[i] = Ops::mul(s, t[i]);
        return r;
    }
    // value fv with derivatives da, db with respect to *this and b: tangents da * t + db * b.t
    __device__ __forceinline__ Dual chain2(R fv, R da, const Dual& b, R db) const {
        Dual r;
        r.v = fv;
        const T sa = Ops::splat(da), sb = Ops::splat(db);
#pragma unroll
        for (int i = 0; i < L; ++i) r.t[i] = Ops::fma(sa, t[i], Ops::mul(sb, b.t[i]));
        return r;
    }
    // the quotient q = *this / b with rb = 1 / b: tangents (t - q b.t) rb
    __device__ __forceinline__ Dual quotient(R q, R rb, const Dual& b) const {
        Dual r;
        r.v = q;
        const T nq = Ops::splat(-q), s = Ops::splat(rb);
#pragma unroll
        for (int i = 0; i < L; ++i) r.t[i] = Ops::mul(Ops::fma(nq, b.t[i], t[i]), s);
        return r;
    }

    __device__ __forceinline__ Dual& operator+=(const Dual& b) { return *this = *this + b; }
    __device__ __forceinline__ Dual& operator-=(const Dual& b) { return *this = *this - b; }
    __device__ __forceinline__ Dual& operator*=(const Dual& b) { return *this = *this * b; }
    __device__ __forceinline__ Dual& operator/=(const Dual& b) { return *this = *this / b; }
    template <typename A, if_arith<A> = 0>
    __device__ __forceinline__ Dual& operator+=(A b) { return *this = *this + b; }
    template <typename A, if_arith<A> = 0>
    __device__ __forceinline__ Dual& operator-=(A b) { return *this = *this - b; }
    template <typename A, if_arith<A> = 0>
    __device__ __forceinline__ Dual& operator*=(A b) { return *this = *this * b; }
    template <typename A, if_arith<A> = 0>
    __device__ __forceinline__ Dual& operator/=(A b) { return *this = *this / b; }
};

// ------------------------------------------------------------------------------------------------
// arithmetic
// ------------------------------------------------------------------------------------------------
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> operator-(const Dual<R, K>& a) {
    Dual<R, K> r;
    r.v = -a.v;
#pragma unroll
    for (int i = 0; i < Dual<R, K>::L; ++i) r.t[i] = Tan<R>::neg(a.t[i]);
    return r;
}

template <typename R, int K>
__device__ __forceinline__ Dual<R, K> operator+(const Dual<R, K>& a, const Dual<R, K>& b) {
    Dual<R, K> r;
    r.v = a.v + b.v;
#pragma unroll
    for (int i = 0; i < Dual<R, K>::L; ++i) r.t[i] = Tan<R>::add(a.t[i], b.t[i]);
    return r;
}

template <typename R, int K>
__device__ __forceinline__ Dual<R, K> operator-(const Dual<R, K>& a, const Dual<R, K>& b) {
    Dual<R, K> r;
    r.v = a.v - b.v;
#pragma unroll
    for (int i = 0; i < Dual<R, K>::L; ++i) r.t[i] = Tan<R>::sub(a.t[i], b.t[i]);
    return r;
}

template <typename R, int K>
__device__ __forceinline__ Dual<R, K> operator*(const Dual<R, K>& a, const Dual<R, K>& b) {
    return a.chain2(a.v * b.v, b.v, b, a.v);
}

template <typename R, int K>
__device__ __forceinline__ Dual<R, K> operator/(const Dual<R, K>& a, const Dual<R, K>& b) {
    return a.quotient(a.v / b.v, R(1) / b.v, b);
}

template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator+(const Dual<R, K>& a, A b) {
    Dual<R, K> r = a;
    r.v = a.v + R(b);
    return r;
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator+(A a, const Dual<R, K>& b) {
    Dual<R, K> r = b;
    r.v = R(a) + b.v;
    return r;
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator-(const Dual<R, K>& a, A b) {
    Dual<R, K> r = a;
    r.v = a.v - R(b);
    return r;
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator-(A a, const Dual<R, K>& b) {
    Dual<R, K> r = -b;
    r.v = R(a) - b.v;
    return r;
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator*(const Dual<R, K>& a, A b) {
    return a.chain(a.v * R(b), R(b));
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator*(A a, const Dual<R, K>& b) {
    return b.chain(R(a) * b.v, R(a));
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator/(const Dual<R, K>& a, A b) {
    return a.chain(a.v / R(b), R(1) / R(b));
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> operator/(A a, const Dual<R, K>& b) {
    const R q = R(a) / b.v;
    return b.chain(q, -q / b.v);
}

// ------------------------------------------------------------------------------------------------
// comparisons: on the values
// ------------------------------------------------------------------------------------------------
#define IRS_AD_COMPARE(OP)                                                                              \
    template <typename R, int K>                                                                        \
    __device__ __forceinline__ bool operator OP(const Dual<R, K>& a, const Dual<R, K>& b) {             \
        return a.v OP b.v;                                                                              \
    }                                                                                                   \
    template <typename R, int K, typename A, if_arith<A> = 0>                                           \
    __device__ __forceinline__ bool operator OP(const Dual<R, K>& a, A b) { return a.v OP R(b); }       \
    template <typename R, int K, typename A, if_arith<A> = 0>                                           \
    __device__ __forceinline__ bool operator OP(A a, const Dual<R, K>& b) { return R(a) OP b.v; }
IRS_AD_COMPARE(<)
IRS_AD_COMPARE(<=)
IRS_AD_COMPARE(>)
IRS_AD_COMPARE(>=)
IRS_AD_COMPARE(==)
IRS_AD_COMPARE(!=)
#undef IRS_AD_COMPARE

// ------------------------------------------------------------------------------------------------
// elementary functions.  The values are libdevice's float and double functions (what a plain body calls);
// the derivatives are formed from them.
// ------------------------------------------------------------------------------------------------
namespace fn {
#define IRS_AD_FN(NAME, FNAME)                                                               \
    __device__ __forceinline__ float NAME(float a) { return ::FNAME(a); }                    \
    __device__ __forceinline__ double NAME(double a) { return ::NAME(a); }
IRS_AD_FN(sqrt, sqrtf)
IRS_AD_FN(exp, expf)
IRS_AD_FN(log, logf)
IRS_AD_FN(sin, sinf)
IRS_AD_FN(cos, cosf)
IRS_AD_FN(tan, tanf)
IRS_AD_FN(asin, asinf)
IRS_AD_FN(acos, acosf)
IRS_AD_FN(atan, atanf)
IRS_AD_FN(sinh, sinhf)
IRS_AD_FN(cosh, coshf)
IRS_AD_FN(tanh, tanhf)
#undef IRS_AD_FN
__device__ __forceinline__ void sincos(float a, float* s, float* c) { ::sincosf(a, s, c); }
__device__ __forceinline__ void sincos(double a, double* s, double* c) { ::sincos(a, s, c); }
__device__ __forceinline__ float atan2(float y, float x) { return ::atan2f(y, x); }
__device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
__device__ __forceinline__ float pow(float a, float e) { return ::powf(a, e); }
__device__ __forceinline__ double pow(double a, double e) { return ::pow(a, e); }
}  // namespace fn

template <typename R, int K>
__device__ __forceinline__ Dual<R, K> sqrt(const Dual<R, K>& a) {
    const R r = fn::sqrt(a.v);
    return a.chain(r, R(0.5) / r);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> exp(const Dual<R, K>& a) {
    const R e = fn::exp(a.v);
    return a.chain(e, e);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> log(const Dual<R, K>& a) {
    return a.chain(fn::log(a.v), R(1) / a.v);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> sin(const Dual<R, K>& a) {
    R s, c;
    fn::sincos(a.v, &s, &c);
    return a.chain(s, c);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> cos(const Dual<R, K>& a) {
    R s, c;
    fn::sincos(a.v, &s, &c);
    return a.chain(c, -s);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> tan(const Dual<R, K>& a) {
    const R t = fn::tan(a.v);
    return a.chain(t, R(1) + t * t);
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> asin(const Dual<R, K>& a) {
    return a.chain(fn::asin(a.v), R(1) / fn::sqrt(R(1) - a.v * a.v));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> acos(const Dual<R, K>& a) {
    return a.chain(fn::acos(a.v), R(-1) / fn::sqrt(R(1) - a.v * a.v));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> atan(const Dual<R, K>& a) {
    return a.chain(fn::atan(a.v), R(1) / (R(1) + a.v * a.v));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> atan2(const Dual<R, K>& y, const Dual<R, K>& x) {
    const R ir2 = R(1) / (x.v * x.v + y.v * y.v);
    return y.chain2(fn::atan2(y.v, x.v), x.v * ir2, x, -y.v * ir2);
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> atan2(const Dual<R, K>& y, A x) {
    const R xv = R(x);
    return y.chain(fn::atan2(y.v, xv), xv / (xv * xv + y.v * y.v));
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> atan2(A y, const Dual<R, K>& x) {
    const R yv = R(y);
    return x.chain(fn::atan2(yv, x.v), -yv / (x.v * x.v + yv * yv));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> sinh(const Dual<R, K>& a) {
    return a.chain(fn::sinh(a.v), fn::cosh(a.v));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> cosh(const Dual<R, K>& a) {
    return a.chain(fn::cosh(a.v), fn::sinh(a.v));
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> tanh(const Dual<R, K>& a) {
    const R t = fn::tanh(a.v);
    return a.chain(t, R(1) - t * t);
}
// |a|: the + branch at 0
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> fabs(const Dual<R, K>& a) {
    return a.v >= R(0) ? a : -a;
}
// the selected argument, value and tangent; the first one on a tie
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> fmin(const Dual<R, K>& a, const Dual<R, K>& b) {
    return b.v < a.v ? b : a;
}
template <typename R, int K>
__device__ __forceinline__ Dual<R, K> fmax(const Dual<R, K>& a, const Dual<R, K>& b) {
    return b.v > a.v ? b : a;
}
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> fmin(const Dual<R, K>& a, A b) { return fmin(a, Dual<R, K>(b)); }
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> fmin(A a, const Dual<R, K>& b) { return fmin(Dual<R, K>(a), b); }
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> fmax(const Dual<R, K>& a, A b) { return fmax(a, Dual<R, K>(b)); }
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> fmax(A a, const Dual<R, K>& b) { return fmax(Dual<R, K>(a), b); }
// a^e for a constant exponent
template <typename R, int K, typename A, if_arith<A> = 0>
__device__ __forceinline__ Dual<R, K> pow(const Dual<R, K>& a, A e) {
    const R er = R(e);
    return a.chain(fn::pow(a.v, er), er * fn::pow(a.v, er - R(1)));
}

}  // namespace ad

// Math<> of a dual number: the value is Math<R>'s (float keeps its fast intrinsics), the derivative is
// formed from that value.
template <typename R, int K>
struct Math<ad::Dual<R, K>> {
    using D = ad::Dual<R, K>;
    static __device__ __forceinline__ void sincos(const D& a, D& s, D& c) {
        R sv, cv;
        Math<R>::sincos(a.v, sv, cv);
        s = a.chain(sv, cv);
        c = a.chain(cv, -sv);
    }
    static __device__ __forceinline__ D rcp(const D& a) {
        const R r = Math<R>::rcp(a.v);
        return a.chain(r, -r * r);
    }
    static __device__ __forceinline__ D div(const D& a, const D& b) {
        return a.quotient(Math<R>::div(a.v, b.v), Math<R>::rcp(b.v), b);
    }
};

}  // namespace irs
