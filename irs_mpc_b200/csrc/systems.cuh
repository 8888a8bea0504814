// __device__ functors for the four analytic systems of the reference and its learned (MLP) dynamics, templated on the scalar
// type R (float for the T x N sample work, double for the sequential rollouts).
//
// Interface (all static-shape, everything stays in registers after unrolling):
//   N, M, D=N+M          state / input / regressor dimensions
//   NJ                   number of Jacobian scalars that vary with (x,u)
//   step<BATCH>(x,u,o)   o = f(x,u).  BATCH selects the reference's `dynamics_batch` semantics
//                        where it differs from the scalar `dynamics` (three_cart only)
//   jac_var(x,u,v)       the NJ varying scalars of d f / d(x,u)
//   jac_assemble(v,J)    J[N*D] (row-major, A|B column order, dynamical_system.py:41-43) from v;
//                        affine in v, so mean(J) == assemble(mean(v))
//   project(x)           non-penetration projection of a sample (three_cart); no-op otherwise
#pragma once
#include <type_traits>

#include "common.cuh"

namespace irs {

#ifndef IRS_USER_SYSTEM
enum SystemId { kPendulum = 0, kBicycle = 1, kQuadrotor = 2, kThreeCart = 3, kMlp21 = 4, kNumSystems = 5 };
#else
// A library built around one user-written system (irs_mpc_b200/user_system.py generates the translation
// unit): its functor is irs::UserSystem<R>, defined after this header with IRS_USER_N states, IRS_USER_M
// inputs and IRS_USER_NPARAMS parameters (h first).  The system dispatch of such a library holds that system
// alone.
enum SystemId { kPendulum = 0, kBicycle = 1, kQuadrotor = 2, kThreeCart = 3, kMlp21 = 4, kUser = 5, kNumSystems = 6 };
template <typename R>
struct UserSystem;
#endif

// ---------------------------------------------------------------------------------------------
// parameter i in the functor's scalar type: fp32 reads the host-rounded mirror
template <typename R>
__device__ __forceinline__ R prm(const SysParams& p, int i) {
    if constexpr (std::is_same<R, float>::value) return p.f[i];
    else return R(p.v[i]);
}

// ---------------------------------------------------------------------------------------------
// Pendulum — examples/pendulum/pendulum_dynamics.py:46-81 (dynamics), :110-127 (Jacobian).
// params: [h]
// ---------------------------------------------------------------------------------------------
template <typename R>
struct Pendulum {
    template <typename S> using Rebind = Pendulum<S>;
    static constexpr int N = 2, M = 1, D = 3, NJ = 1;
    static constexpr bool kHasJacobian = true;
    static constexpr int kTrigAhead = 0;
    static constexpr bool kHasProjection = false;
    R h;
    __device__ explicit Pendulum(const SysParams& p) : h(prm<R>(p, 0)) {}

    template <bool BATCH>
    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {
        R s, c;
        Math<R>::sincos(x[0], s, c);
        const R v = x[1] + h * (u[0] - s);      // semi-implicit Euler (:55-57)
        o[1] = v;
        o[0] = x[0] + h * v;
    }
    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* v) const {
        R s, c;
        Math<R>::sincos(x[0], s, c);
        v[0] = c;
    }
    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {
        J[0] = R(1) - h * h * v[0];  J[1] = h;     J[2] = h * h;
        J[3] = -h * v[0];            J[4] = R(1);  J[5] = h;
    }
    __device__ __forceinline__ void project(R* x) const {}
};

// ---------------------------------------------------------------------------------------------
// Bicycle — examples/bicycle/bicycle_dynamics.py:47-86 (dynamics), :115-132 (Jacobian).
// x = [px, py, heading, speed, steer], u = [accel, steer rate].  params: [h]
// ---------------------------------------------------------------------------------------------
template <typename R>
struct Bicycle {
    template <typename S> using Rebind = Bicycle<S>;
    static constexpr int N = 5, M = 2, D = 7, NJ = 6;
    static constexpr bool kHasJacobian = true;
    static constexpr int kTrigAhead = 0;
    static constexpr bool kHasProjection = false;
    R h;
    __device__ explicit Bicycle(const SysParams& p) : h(prm<R>(p, 0)) {}

    template <bool BATCH>
    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {
        R s, c, sd, cd;
        Math<R>::sincos(x[2], s, c);
        Math<R>::sincos(x[4], sd, cd);
        const R v = x[3];
        o[0] = x[0] + h * (v * c);
        o[1] = x[1] + h * (v * s);
        o[2] = x[2] + h * (v * Math<R>::div(sd, cd));
        o[3] = x[3] + h * u[0];
        o[4] = x[4] + h * u[1];
    }
    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* v) const {
        R s, c, sd, cd;
        Math<R>::sincos(x[2], s, c);
        Math<R>::sincos(x[4], sd, cd);
        const R icd = Math<R>::rcp(cd);
        v[0] = x[3] * s;          // -> J[0][2] = -h v sin(th)
        v[1] = c;                 // -> J[0][3] =  h cos(th)
        v[2] = x[3] * c;          // -> J[1][2] =  h v cos(th)
        v[3] = s;                 // -> J[1][3] =  h sin(th)
        v[4] = sd * icd;          // -> J[2][3] =  h tan(de)
        v[5] = x[3] * icd * icd;  // -> J[2][4] =  h v / cos^2(de)
    }
    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {
#pragma unroll
        for (int i = 0; i < N * D; ++i) J[i] = R(0);
#pragma unroll
        for (int i = 0; i < N; ++i) J[i * D + i] = R(1);
        J[0 * D + 2] = -h * v[0];
        J[0 * D + 3] = h * v[1];
        J[1 * D + 2] = h * v[2];
        J[1 * D + 3] = h * v[3];
        J[2 * D + 3] = h * v[4];
        J[2 * D + 4] = h * v[5];
        J[3 * D + 5] = h;
        J[4 * D + 6] = h;
    }
    __device__ __forceinline__ void project(R* x) const {}
};

// ---------------------------------------------------------------------------------------------
// Quadrotor — examples/quadrotor/quadrotor_dynamics.py:40-77 with helpers :150-231.
// x = [xyz, rpy, xyz_dot, rpy_dot], u = 4 rotor commands.
// params: [h, mass, L, g, Ixx, Iyy, Izz, kF, kM]  (defaults :26-38)
// ---------------------------------------------------------------------------------------------
#include "quadrotor_jac.inc"

template <typename R>
struct Quadrotor {
    template <typename S> using Rebind = Quadrotor<S>;
    static constexpr int N = 12, M = 4, D = 16, NJ = IRS_QUAD_NJ;
    static constexpr bool kHasJacobian = true;
    static constexpr bool kHasProjection = false;
    R h, mass, L, g, I0, I1, I2, kF, kM;
    // loop invariants (fp32: computed on the host in double precision, SysParams::f[9..16])
    R inv_mass, inv_I0, inv_I1, inv_I2, LkF, dI12, dI20, dI01;
    __device__ explicit Quadrotor(const SysParams& p)
        : h(prm<R>(p, 0)), mass(prm<R>(p, 1)), L(prm<R>(p, 2)), g(prm<R>(p, 3)), I0(prm<R>(p, 4)),
          I1(prm<R>(p, 5)), I2(prm<R>(p, 6)), kF(prm<R>(p, 7)), kM(prm<R>(p, 8)) {
        if constexpr (std::is_same<R, float>::value) {
            inv_mass = p.f[9];  inv_I0 = p.f[10];  inv_I1 = p.f[11];  inv_I2 = p.f[12];
            LkF = p.f[13];  dI12 = p.f[14];  dI20 = p.f[15];  dI01 = p.f[16];
        } else {
            inv_mass = R(1.0 / p.v[1]);  inv_I0 = R(1.0 / p.v[4]);  inv_I1 = R(1.0 / p.v[5]);
            inv_I2 = R(1.0 / p.v[6]);  LkF = L * kF;  dI12 = I1 - I2;  dI20 = I2 - I0;  dI01 = I0 - I1;
        }
    }

    // The Euler angles of the NEXT state, x[3+j] + h x[9+j], do not depend on the input: their sines
    // and cosines can be evaluated one step ahead, off the sequential path of a rollout
    // (tvlqr.cuh: rollout_trig_kernel).  sc = {sin r, cos r, sin p, cos p, sin y, cos y}.
    static constexpr int kTrigAhead = 3;
    // (explicit fma: the rollout's helper warp and its recursion evaluate this in different contexts and
    //  must round identically)
    __device__ __forceinline__ R next_angle(R angle, R rate) const { return fma(h, rate, angle); }
    static __device__ __forceinline__ void trig(R angle, R& s, R& c) { Math<R>::sincos(angle, s, c); }

    template <bool BATCH>
    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {
        R sc[6];
        Math<R>::sincos(x[3], sc[0], sc[1]);
        Math<R>::sincos(x[4], sc[2], sc[3]);
        Math<R>::sincos(x[5], sc[4], sc[5]);
        step_trig<BATCH>(x, u, sc, o);
    }
    // Both members of an antithetic pair at once, x = (x̄ + z, x̄ − z) in the two halves of every float2
    // (smooth_tc.cuh, kTcPaired): each half gets the bits step<false> gives that member alone.
    __device__ __forceinline__ void step_pair(const float2* x, const float2* u, float2* o) const {
        float2 sc[6];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            Math<float>::sincos(x[3 + j].x, sc[2 * j].x, sc[2 * j + 1].x);
            Math<float>::sincos(x[3 + j].y, sc[2 * j].y, sc[2 * j + 1].y);
        }
        step_lanes(x, u, sc, o);
    }
    template <bool BATCH>
    __device__ __forceinline__ void step_trig(const R* x, const R* u, const R* sc, R* o) const {
        if constexpr (std::is_same<R, float>::value) step_lanes(x, u, sc, o);
        else step_trig_fp64(x, u, sc, o);
    }
    // The fp32 step on one sample (V = float) or on two (V = float2), every rounding explicit: the
    // contractions are those nvcc chose for the expression form below, so both keep their former bits.
    template <typename V>
    __device__ __forceinline__ void step_lanes(const V* x, const V* u, const V* sc, V* o) const {
        using L = Lanes<V>;
        const V sr = sc[0], cr = sc[1], sp = sc[2], cp = sc[3], sy = sc[4], cy = sc[5];
        const V icp = L::rcp(cp);
        const V rd0 = x[9], rd1 = x[10], rd2 = x[11];
        const V hh = L::splat(h);
        const V s03 = L::add(u[0], u[3]), s12 = L::add(u[1], u[2]);
        const V Fz = L::mul(L::splat(kF), L::add(s03, s12));
        const V M0 = L::mul(L::splat(LkF), L::sub(L::add(u[2], u[3]), L::add(u[0], u[1])));
        const V M1 = L::mul(L::splat(LkF), L::sub(s12, s03));
        const V M2 = L::mul(L::splat(kM), L::sub(L::add(u[1], u[3]), L::add(u[0], u[2])));
        const V a = L::mul(Fz, L::splat(inv_mass));
        const V spcr = L::mul(sp, cr);
        o[6] = L::fma(hh, L::mul(a, L::fma(sy, sr, L::mul(cy, spcr))), x[6]);
        o[7] = L::fma(hh, L::mul(a, L::fma(sy, spcr, L::neg(L::mul(cy, sr)))), x[7]);
        o[8] = L::fma(hh, L::fma(a, L::mul(cp, cr), L::splat(-g)), x[8]);
        const V cprd2 = L::mul(cp, rd2);
        const V p = L::fma(L::neg(sp), rd2, rd0);
        const V q = L::fma(cr, rd1, L::mul(sr, cprd2));
        const V r = L::fma(cr, cprd2, L::neg(L::mul(sr, rd1)));
        const V pd_I0 = L::fma(L::splat(dI12), L::mul(q, r), M0);       // pd * I0
        const V qd = L::mul(L::fma(L::splat(dI20), L::mul(r, p), M1), L::splat(inv_I1));
        const V rdd = L::mul(L::fma(L::splat(dI01), L::mul(p, q), M2), L::splat(inv_I2));
        const V tp = L::mul(sp, icp);
        const V icp2 = L::mul(icp, icp);
        const V srq_crr = L::fma(sr, q, L::mul(cr, r));
        const V crq_srr = L::fma(cr, q, L::neg(L::mul(sr, r)));
        const V srqd_crrd = L::fma(sr, qd, L::mul(cr, rdd));
        o[9] = L::fma(hh, L::fma(rd1, L::mul(icp2, srq_crr),
                                 L::fma(rd0, L::mul(tp, crq_srr), L::fma(pd_I0, L::splat(inv_I0), L::mul(tp, srqd_crrd)))),
                      x[9]);
        o[10] = L::fma(hh, L::fma(L::neg(rd0), srq_crr, L::fma(cr, qd, L::neg(L::mul(sr, rdd)))), x[10]);
        o[11] = L::fma(hh, L::fma(rd1, L::mul(L::mul(tp, icp), srq_crr), L::fma(rd0, L::mul(icp, crq_srr), L::mul(icp, srqd_crrd))),
                       x[11]);
#pragma unroll
        for (int i = 0; i < 6; ++i) o[i] = L::fma(hh, x[6 + i], x[i]);     // kinematics; next_angle for i >= 3
    }
    __device__ __forceinline__ void step_trig_fp64(const R* x, const R* u, const R* sc, R* o) const {
        const R sr = sc[0], cr = sc[1], sp = sc[2], cp = sc[3], sy = sc[4], cy = sc[5];
        const R icp = Math<R>::rcp(cp);
        const R rd0 = x[9], rd1 = x[10], rd2 = x[11];
        // thrust and moments (:43-49)
        const R s03 = u[0] + u[3], s12 = u[1] + u[2];
        const R Fz = kF * (s03 + s12);
        const R M0 = LkF * ((u[2] + u[3]) - (u[0] + u[1]));
        const R M1 = LkF * (s12 - s03);
        const R M2 = kM * ((u[1] + u[3]) - (u[0] + u[2]));
        // translational acceleration: third column of Rz Ry Rx times Fz (:51-54, :150-189)
        const R a = Fz * inv_mass;
        const R spcr = sp * cr;
        o[6] = x[6] + h * (a * (cy * spcr + sy * sr));
        o[7] = x[7] + h * (a * (sy * spcr - cy * sr));
        o[8] = x[8] + h * (a * (cp * cr) - g);
        // body rates pqr = PhiInv rpy_d (:57-58, :191-202)
        const R cprd2 = cp * rd2;
        const R p = rd0 - sp * rd2;
        const R q = cr * rd1 + sr * cprd2;
        const R r = cr * cprd2 - sr * rd1;
        // pqr_d = I^-1 (M - pqr x I pqr) (:59)
        const R pd = (M0 + dI12 * (q * r)) * inv_I0;
        const R qd = (M1 + dI20 * (r * p)) * inv_I1;
        const R rdd = (M2 + dI01 * (p * q)) * inv_I2;
        // rpy_dd = Phi pqr_d + (dPhi/dt) pqr (:61-68, :204-231)
        const R tp = sp * icp;
        const R icp2 = icp * icp;
        const R srq_crr = sr * q + cr * r;       // appears in Phi rows 0 and 2
        const R crq_srr = cr * q - sr * r;
        const R srqd_crrd = sr * qd + cr * rdd;
        o[9] = x[9] + h * (pd + tp * srqd_crrd + rd0 * (tp * crq_srr) + rd1 * (icp2 * srq_crr));
        o[10] = x[10] + h * ((cr * qd - sr * rdd) - rd0 * srq_crr);
        o[11] = x[11] + h * (icp * srqd_crrd + rd0 * (icp * crq_srr) + rd1 * (tp * icp * srq_crr));
        // kinematics (:70)
#pragma unroll
        for (int i = 0; i < 3; ++i) o[i] = x[i] + h * x[6 + i];
#pragma unroll
        for (int i = 3; i < 6; ++i) o[i] = next_angle(x[i], x[6 + i]);
    }
    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* v) const {
        R sr, cr, sp, cp, sy, cy;
        Math<R>::sincos(x[3], sr, cr);
        Math<R>::sincos(x[4], sp, cp);
        Math<R>::sincos(x[5], sy, cy);
        const R icp = Math<R>::rcp(cp);
        const R rd0 = x[9], rd1 = x[10], rd2 = x[11];
        const R u0 = u[0], u1 = u[1], u2 = u[2], u3 = u[3];
        IRS_QUAD_JAC_BODY(v)
    }
    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {
        constexpr int rows[NJ] = IRS_QUAD_JAC_ROWS;
        constexpr int cols[NJ] = IRS_QUAD_JAC_COLS;
#pragma unroll
        for (int i = 0; i < N * D; ++i) J[i] = R(0);
#pragma unroll
        for (int i = 0; i < N; ++i) J[i * D + i] = R(1);
#pragma unroll
        for (int i = 0; i < 6; ++i) J[i * D + 6 + i] = h;
#pragma unroll
        for (int k = 0; k < NJ; ++k) J[rows[k] * D + cols[k]] += h * v[k];
    }
    __device__ __forceinline__ void project(R* x) const {}
};

// ---------------------------------------------------------------------------------------------
// Three carts — examples/three_cart/three_cart_dynamics.py.
// x = [q1,q2,q3,v1,v2,v3], u = [u1,u3].  params: [h, cart width d]
//   step<false>: scalar `dynamics` (:22-107): pair collisions push out by HALF the depth
//   step<true> : `dynamics_batch` (:109-194): pair collisions push out by the FULL depth
//   project    : `projection` (:196-264), half depth, positions only
// The gap tests use explicit subtract-then-compare (no contraction) so that the case a sample
// falls in is a pure function of the rounded free-step state.
// ---------------------------------------------------------------------------------------------
template <typename R>
struct ThreeCart {
    template <typename S> using Rebind = ThreeCart<S>;
    static constexpr int N = 6, M = 2, D = 8, NJ = 0;
    static constexpr bool kHasJacobian = false;   // three_cart_dynamics.py:20
    static constexpr int kTrigAhead = 0;
    static constexpr bool kHasProjection = true;
    static constexpr int kProjDims = 3;           // project() touches the cart positions only
    R h, d;
    __device__ explicit ThreeCart(const SysParams& p) : h(prm<R>(p, 0)), d(prm<R>(p, 1)) {}

    // case id: 0 none, 1 all three, 2 carts 1-2, 3 carts 2-3  (:146-157)
    __device__ __forceinline__ int contact_case(R q1, R q2, R q3) const {
        const bool g12 = (q2 - q1) < d;
        const bool g23 = (q3 - q2) < d;
        return g12 ? (g23 ? 1 : 2) : (g23 ? 3 : 0);
    }
    // Branch-free (selects): the four contact cases are exclusive, every candidate value is computed and
    // the case picks; each selected value is produced by the same operations as in the reference's
    // branch, so the results are bit-identical to a branching version while a warp whose lanes fall into
    // different cases does not serialise them (and the compiler can interleave independent samples).
    template <bool BATCH>
    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {
        const R v1 = x[3] + h * u[0];
        const R v2 = x[4];
        const R v3 = x[5] + h * u[1];
        const R q1 = x[0] + h * v1;
        const R q2 = x[1] + h * v2;
        const R q3 = x[2] + h * v3;
        const R gap12 = q2 - q1, gap23 = q3 - q2;
        const bool g12 = gap12 < d, g23 = gap23 < d;
        const bool all3 = g12 && g23, pair12 = g12 && !g23, pair23 = !g12 && g23;      // cases 1, 2, 3 (:146-157)
        const R pf = BATCH ? R(1) : R(0.5);
        const R mid = (q1 + q2 + q3) * R(1.0 / 3.0);
        const R va3 = (v1 + v2 + v3) * R(1.0 / 3.0);
        const R depth12 = pf * (d - gap12), va12 = R(0.5) * (v1 + v2);
        const R depth23 = pf * (d - gap23), va23 = R(0.5) * (v2 + v3);
        o[0] = all3 ? mid - d : (pair12 ? q1 - depth12 : q1);
        o[1] = all3 ? mid : (pair12 ? q2 + depth12 : (pair23 ? q2 - depth23 : q2));
        o[2] = all3 ? mid + d : (pair23 ? q3 + depth23 : q3);
        o[3] = all3 ? va3 : (pair12 ? va12 : v1);
        o[4] = all3 ? va3 : (pair12 ? va12 : (pair23 ? va23 : v2));
        o[5] = all3 ? va3 : (pair23 ? va23 : v3);
    }
    __device__ __forceinline__ void jac_var(const R*, const R*, R*) const {}
    __device__ __forceinline__ void jac_assemble(const R*, R*) const {}
    __device__ __forceinline__ void project(R* x) const {
        // sequential masks as in :216-261 (each re-evaluated on the partially projected point), written
        // with selects: the operations that produce a selected value are those of the reference's branch
        R x0 = x[0], x1 = x[1], x2 = x[2];
        {
            const bool c = (x1 - x0) < d && (x2 - x1) < d;
            const R mid = (x0 + x1 + x2) * R(1.0 / 3.0);
            const R lo = mid - d, hi = mid + d;
            x1 = c ? mid : x1;  x0 = c ? lo : x0;  x2 = c ? hi : x2;
        }
        {
            const R gap = x1 - x0;
            const bool c = gap < d && !((x2 - x1) < d);
            const R depth = R(0.5) * (d - gap);
            const R up = x1 + depth, dn = x0 - depth;
            x1 = c ? up : x1;  x0 = c ? dn : x0;
        }
        {
            const R gap = x2 - x1;
            const bool c = !((x1 - x0) < d) && gap < d;
            const R depth = R(0.5) * (d - gap);
            const R up = x2 + depth, dn = x1 - depth;
            x2 = c ? up : x2;  x1 = c ? dn : x1;
        }
        x[0] = x0;  x[1] = x1;  x[2] = x2;
    }
};

// Centred accumulation (smooth.cuh: kFlagCentered): the regressors of nominal point (xbar, ubar) are the
// absolute points xbar + z', so the state of a sample is 2 xbar + z'.  centred_frame() returns the fp32
// point (xf, uf) such that the kernel evaluates f(xf + z'_x, uf + z'_u) - f(xf, uf): the doubled nominal,
// expressed — where the dynamics allow it — in a frame in which fp32 still resolves what the dynamics
// branch on.  three_cart is equivariant under a common shift of the positions and of the velocities, so
// its frame moves with cart 1: positions and velocities relative to cart 1's (doubled) nominal.  The
// response DIFFERENCE is the same in exact arithmetic, but the contact gaps (O(1)) are no longer computed
// as differences of fp32 numbers of size 2 |xbar|, whose rounding flips the discontinuous velocity merge
// for samples within ulp(2 |xbar|) of a contact threshold.
template <class Sys>
__device__ __forceinline__ void centred_frame(const double* xb, const double* ub, float* xf, float* uf) {
    constexpr int n = Sys::N, m = Sys::M;
    if constexpr (Sys::kHasProjection) {      // ThreeCart
        static_assert(n == 6 && m == 2, "three_cart layout");
        xf[0] = 0.f;
        xf[1] = (float)(2.0 * (xb[1] - xb[0]));
        xf[2] = (float)(2.0 * (xb[2] - xb[0]));
        xf[3] = 0.f;
        xf[4] = (float)(2.0 * (xb[4] - xb[3]));
        xf[5] = (float)(2.0 * (xb[5] - xb[3]));
    } else {
#pragma unroll
        for (int q = 0; q < n; ++q) xf[q] = (float)(2.0 * xb[q]);
    }
#pragma unroll
    for (int q = 0; q < m; ++q) uf[q] = (float)(2.0 * ub[q]);
}

// ---------------------------------------------------------------------------------------------
// Learned dynamics — examples/pendulum/pendulum_nn.py:19-33 (network), :66-90 (the DynamicalSystem
// wrapper): x+ = net([x, u]) with net = Linear(d, H1) ReLU Linear(H1, H2) ReLU Linear(H2, n), float32
// (the reference evaluates the torch module on float32 tensors and returns float32).  The Jacobian is
// the exact derivative of the piecewise-linear network, W3 diag(a2 > 0) W2 diag(a1 > 0) W1, which is
// what torch.autograd returns in pendulum_nn.py:78-85.
// This per-thread functor serves every generic kernel (dynamics / Jacobian batches, rollouts, first-order
// smoothing, the fp64 nominal point of the fit); the T x N zero-order sample work runs the hidden layer on
// the tensor cores instead (smooth_mlp.cuh).
// blob (float32): W1[H1][d] | b1[H1] | W2[H2][H1] | b2[H2] | W3[n][H2] | b3[n] | W2^T[H1][H2] (for the warp-cooperative
// step of the rollouts: lanes over units read it coalesced); registered with irs_mlp_register.
// params: [h, handle]
// ---------------------------------------------------------------------------------------------
constexpr int kMlpMaxHidden = 128;

struct MlpView {
    const float *w1, *b1, *w2, *b2, *w3, *b3, *w2t;
    int H1, H2;
    __host__ __device__ MlpView(const float* blob, int d, int n, int h1, int h2) : H1(h1), H2(h2) {
        w1 = blob;          b1 = w1 + h1 * d;
        w2 = b1 + h1;       b2 = w2 + h2 * h1;
        w3 = b2 + h2;       b3 = w3 + n * h2;
        w2t = b3 + n;
    }
    static __host__ __device__ long long floats(int d, int n, int h1, int h2) {
        return (long long)h1 * d + h1 + 2ll * h2 * h1 + h2 + (long long)n * h2 + n;
    }
};

template <typename R, int N_, int M_>
struct Mlp {
    template <typename S> using Rebind = Mlp<S, N_, M_>;
    static constexpr int N = N_, M = M_, D = N_ + M_, NJ = N_ * (N_ + M_);
    static constexpr bool kHasJacobian = true;
    static constexpr int kTrigAhead = 0;
    static constexpr bool kHasProjection = false;
    static constexpr bool kIsMlp = true;
    MlpView net;
    __device__ explicit Mlp(const SysParams& p) : net(p.mlp, D, N, p.h1, p.h2) {}

    // hidden activations of ([x, u]); sums in four interleaved partial chains (the dependent FFMA chain of a
    // 100-term dot product would otherwise be latency bound)
    __device__ __forceinline__ void hidden(const float* in, float* a1, float* a2) const {
        for (int j = 0; j < net.H1; ++j) {
            float s = __ldg(net.b1 + j);
#pragma unroll
            for (int q = 0; q < D; ++q) s = fmaf(__ldg(net.w1 + j * D + q), in[q], s);
            a1[j] = fmaxf(s, 0.f);
        }
        for (int j = 0; j < net.H2; ++j) a2[j] = fmaxf(dot_row(net.w2 + (long long)j * net.H1, a1, net.H1, __ldg(net.b2 + j)), 0.f);
    }
    // sum_q w[q * stride] a[q] + init: the ONE summation order of every float32 evaluation of a unit
    static __device__ __forceinline__ float dot_row(const float* w, const float* a, int len, float init, int stride = 1) {
        float s0 = init, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int q = 0;
        for (; q + 4 <= len; q += 4) {
            s0 = fmaf(__ldg(w + q * stride), a[q], s0);
            s1 = fmaf(__ldg(w + (q + 1) * stride), a[q + 1], s1);
            s2 = fmaf(__ldg(w + (q + 2) * stride), a[q + 2], s2);
            s3 = fmaf(__ldg(w + (q + 3) * stride), a[q + 3], s3);
        }
        for (; q < len; ++q) s0 = fmaf(__ldg(w + q * stride), a[q], s0);
        return (s0 + s1) + (s2 + s3);
    }
    // step() by one warp: every lane holds the same (x, u) and receives o; lanes over the hidden units, each unit
    // summed exactly as in step() (bit-identical result).  a1s, a2s: kMlpMaxHidden floats of shared memory each.
    __device__ __forceinline__ void step_warp(const R* x, const R* u, R* o, float* a1s, float* a2s, int lane) const {
        float in[D];
#pragma unroll
        for (int q = 0; q < N; ++q) in[q] = (float)x[q];
#pragma unroll
        for (int q = 0; q < M; ++q) in[N + q] = (float)u[q];
        for (int j = lane; j < net.H1; j += 32) {
            float s = __ldg(net.b1 + j);
#pragma unroll
            for (int q = 0; q < D; ++q) s = fmaf(__ldg(net.w1 + j * D + q), in[q], s);
            a1s[j] = fmaxf(s, 0.f);
        }
        __syncwarp();
        {   // hidden layer: a lane carries its (up to four) units j = lane + 32 r TOGETHER — sixteen independent FFMA
            // chains instead of four, one pass over the activations; per unit the order of dot_row
            static_assert(kMlpMaxHidden <= 128, "four units per lane");
            float sacc[4][4];
            int col[4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const int j = lane + 32 * r;
                col[r] = j < net.H2 ? j : net.H2 - 1;                      // surplus lanes shadow the last unit
                sacc[r][0] = __ldg(net.b2 + col[r]);
                sacc[r][1] = sacc[r][2] = sacc[r][3] = 0.f;
            }
            int q = 0;
            for (; q + 4 <= net.H1; q += 4) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float av = a1s[q + c];
                    const float* wrow = net.w2t + (long long)(q + c) * net.H2;
#pragma unroll
                    for (int r = 0; r < 4; ++r) sacc[r][c] = fmaf(__ldg(wrow + col[r]), av, sacc[r][c]);
                }
            }
            for (; q < net.H1; ++q) {
                const float av = a1s[q];
#pragma unroll
                for (int r = 0; r < 4; ++r) sacc[r][0] = fmaf(__ldg(net.w2t + (long long)q * net.H2 + col[r]), av, sacc[r][0]);
            }
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (lane + 32 * r < net.H2) a2s[lane + 32 * r] = fmaxf((sacc[r][0] + sacc[r][1]) + (sacc[r][2] + sacc[r][3]), 0.f);
        }
        __syncwarp();
        float mine = 0.f;
        if (lane < N) mine = dot_row(net.w3 + (long long)lane * net.H2, a2s, net.H2, __ldg(net.b3 + lane));
#pragma unroll
        for (int k = 0; k < N; ++k) o[k] = R(__shfl_sync(0xffffffffu, mine, k));
        __syncwarp();      // a1s / a2s may be rewritten by the next call
    }

    template <bool BATCH>
    __device__ __forceinline__ void step(const R* x, const R* u, R* o) const {
        float in[D], a1[kMlpMaxHidden], a2[kMlpMaxHidden];
#pragma unroll
        for (int q = 0; q < N; ++q) in[q] = (float)x[q];
#pragma unroll
        for (int q = 0; q < M; ++q) in[N + q] = (float)u[q];
        hidden(in, a1, a2);
#pragma unroll
        for (int k = 0; k < N; ++k) o[k] = R(dot_row(net.w3 + (long long)k * net.H2, a2, net.H2, __ldg(net.b3 + k)));
    }
    __device__ __forceinline__ void jac_var(const R* x, const R* u, R* v) const {
        float in[D], a1[kMlpMaxHidden], a2[kMlpMaxHidden];
#pragma unroll
        for (int q = 0; q < N; ++q) in[q] = (float)x[q];
#pragma unroll
        for (int q = 0; q < M; ++q) in[N + q] = (float)u[q];
        hidden(in, a1, a2);
        // reverse mode, one output row at a time: r1 = (W3[k] o mask2) W2 o mask1, J[k] = r1 W1
#pragma unroll 1
        for (int k = 0; k < N; ++k) {
            float r1[kMlpMaxHidden];
            for (int j = 0; j < net.H1; ++j) r1[j] = 0.f;
            for (int q = 0; q < net.H2; ++q) {
                if (a2[q] > 0.f) {
                    const float g = __ldg(net.w3 + (long long)k * net.H2 + q);
                    const float* row = net.w2 + (long long)q * net.H1;
                    for (int j = 0; j < net.H1; ++j) r1[j] = fmaf(g, __ldg(row + j), r1[j]);
                }
            }
            float acc[D];
#pragma unroll
            for (int c = 0; c < D; ++c) acc[c] = 0.f;
            for (int j = 0; j < net.H1; ++j) {
                if (a1[j] > 0.f) {
#pragma unroll
                    for (int c = 0; c < D; ++c) acc[c] = fmaf(r1[j], __ldg(net.w1 + j * D + c), acc[c]);
                }
            }
#pragma unroll
            for (int c = 0; c < D; ++c) v[k * D + c] = R(acc[c]);
        }
    }
    __device__ __forceinline__ void jac_assemble(const R* v, R* J) const {
#pragma unroll
        for (int i = 0; i < N * D; ++i) J[i] = v[i];
    }
    __device__ __forceinline__ void project(R* x) const {}
};
template <typename R>
using Mlp21 = Mlp<R, 2, 1>;

template <class Sys>
struct is_mlp : std::false_type {};
template <typename R, int N_, int M_>
struct is_mlp<Mlp<R, N_, M_>> : std::true_type {};

// systems with step_pair (both members of an antithetic pair in packed FP32)
template <class Sys>
struct has_step_pair : std::false_type {};
template <>
struct has_step_pair<Quadrotor<float>> : std::true_type {};

// Host-side dimension table (kept in sync with the functors by static_asserts in api.cu).
struct SystemDims {
    int n, m, nj;
};
inline SystemDims system_dims(int id) {
    switch (id) {
        case kPendulum: return {2, 1, 1};
        case kBicycle: return {5, 2, 6};
        case kQuadrotor: return {12, 4, IRS_QUAD_NJ};
        case kThreeCart: return {6, 2, 0};
        case kMlp21: return {2, 1, 6};
#ifdef IRS_USER_SYSTEM
        case kUser: return {IRS_USER_N, IRS_USER_M, IRS_USER_N * (IRS_USER_N + IRS_USER_M)};
#endif
        default: return {0, 0, 0};
    }
}

// Dispatch a generic lambda-like functor over the system id:  IRS_DISPATCH_SYSTEM(id, R, Sys, {...})
#ifdef IRS_USER_SYSTEM
#define IRS_DISPATCH_SYSTEM(id, R, SYS, ...)                                                        \
    switch (id) {                                                                                   \
        case irs::kUser: { using SYS = irs::UserSystem<R>; __VA_ARGS__; break; }                    \
        default: irs::set_error("this library holds the user system (id %d) only, got id %d", (int)irs::kUser, id); \
                 return 1;                                                                          \
    }
#else
#define IRS_DISPATCH_SYSTEM(id, R, SYS, ...)                                   \
    switch (id) {                                                              \
        case irs::kPendulum: { using SYS = irs::Pendulum<R>; __VA_ARGS__; break; }   \
        case irs::kBicycle: { using SYS = irs::Bicycle<R>; __VA_ARGS__; break; }     \
        case irs::kQuadrotor: { using SYS = irs::Quadrotor<R>; __VA_ARGS__; break; } \
        case irs::kThreeCart: { using SYS = irs::ThreeCart<R>; __VA_ARGS__; break; } \
        case irs::kMlp21: { using SYS = irs::Mlp21<R>; __VA_ARGS__; break; }         \
        default: irs::set_error("unknown system id %d", id); return 1;         \
    }
#endif

}  // namespace irs
