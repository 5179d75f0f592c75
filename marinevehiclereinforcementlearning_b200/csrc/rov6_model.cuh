// BlueROV2 Heavy 6DoF manoeuvring model.  All intermediate state lives in
// registers; the code is written once over a value type V (mvrl_math.cuh):
// float / double = one environment per thread, F2 = two fp32 environments per
// thread on the packed FFMA2 path.  S = VT<V>::S is the scalar type of the
// vehicle constants.  Restates (does not copy) the algorithm of
// dynamicsModel_BlueROV2_Heavy_6DoF.py:220-442 and resources.py:98-143; the
// reference's quirks are kept on purpose (SURVEY.md section 7, "bug-compatibility").
#pragma once
#include <type_traits>
#include "mvrl_math.cuh"

namespace mvrl {

// Constants of one vehicle, converted to the compute type on the host and
// passed to every kernel as a __grid_constant__ argument (constant bank, one
// copy per launch, handle-specific, CUDA-graph friendly).
template <typename T> struct Rov6Dev {
    T m, xg, yg, zg;
    T Ixx, Iyy, Izz, Ixy, Ixz, Iyz;
    T Xud, Yvd, Zwd, Kpd, Mqd, Nrd;
    T Xu, Yv, Yp, Yr, Zw, Zq, Kv, Kp, Kr, Mw, Mq, Nv, Np, Nr;
    T Xuu, Yvv, Ypp, Yrr, Zww, Zqq, Kvv, Kpp, Krr, Mww, Mqq, Nvv, Npp, Nrr;
    T WmB, gx, gy, gz;        // W-B and (xg W - xb B), (yg W - yb B), (zg W - zb B)
    T A[6][8];
    T Ainv[8][6];
    T Minv[6][6];
    T thrust_k;               // thrust_coef / 3600: F = thrust_k * rpm * |rpm|
    T inv_thrust_coef;        // 1 / (rho D^4 Kt)
    T rpm_max, rpm_db;
    T f_max, f_db;            // thruster force at rpm_max / at the deadband edge
    T pKp[6], pKi[6], pKd[6], pWind[6], pMax[6];
    T inv_3L, act_pos, act_ang, inv_ang;  // 1/(3 Length), 2 Length, pi/4, 4/pi
    // Crb + Ca folded for the default sparsity (see body_accel): effective masses
    // m - Xudot.., m*zg, and the differences that multiply the velocity products
    T mX, mY, mZ, mzg, cVW, cUW, cUV, cQR, cPR, cPQ;
    int thrusters_on;
};

template <typename V> struct Trig6 { V sph, cph, sth, cth, sps, cps; };

// fp32 sin/cos without libm's branches: Cody-Waite reduction by pi/2 (three
// FMAs, exact for |x| < 2^16) + the minimax polynomials of the Cephes sinf /
// cosf kernels (|r| <= pi/4, ~1 ulp) + branch-free quadrant fix-up.  Angles are
// wrapped to [0, 2 pi) every env step, so |x| stays far below 2^16; the step
// kernel flags any environment whose unwrapped angle leaves that range in its
// non-finite/out-of-range counter instead of paying a branch per evaluation.
#define MVRL_SINCOS_F32_MAX_ARG 65536.0f

// quadrant fix-up: q = round(x 2/pi) sits in the low mantissa bits of j
__device__ __forceinline__ void sincos_quadrant(float j, float s0, float c0, float* sn, float* cs) {
    const int q = __float_as_int(j);
    const bool swap = (q & 1) != 0;
    const float s1 = swap ? c0 : s0;
    const float c1 = swap ? s0 : c0;
    *sn = __int_as_float(__float_as_int(s1) ^ ((q & 2) << 30));
    *cs = __int_as_float(__float_as_int(c1) ^ (((q + 1) & 2) << 30));
}

// V = float or F2: the arithmetic is shared (packed for F2), the integer fix-up is per lane
template <typename V>
__device__ __forceinline__ void sincos_f32(V x, V* sn, V* cs) {
    const V j = fmaf_t(x, V(0.636619772367581343f), V(12582912.0f));   // round(x * 2/pi) in the low mantissa bits
    const V k = j - V(12582912.0f);
    V r = fmaf_t(k, V(-1.5703125f), x);
    r = fmaf_t(k, V(-4.837512969970703125e-4f), r);
    r = fmaf_t(k, V(-7.549789954891882e-8f), r);
    const V z = r * r;
    V ps = fmaf_t(z, V(-1.9515295891e-4f), V(8.3321608736e-3f));
    ps = fmaf_t(ps, z, V(-1.6666654611e-1f));
    const V s0 = fmaf_t(ps * z, r, r);
    V pc = fmaf_t(z, V(2.443315711809948e-5f), V(-1.388731625493765e-3f));
    pc = fmaf_t(pc, z, V(4.166664568298827e-2f));
    const V c0 = fmaf_t(pc * z, z, fmaf_t(z, V(-0.5f), V(1.0f)));
    if constexpr (VT<V>::L == 1) {
        sincos_quadrant(j, s0, c0, sn, cs);
    } else {
        sincos_quadrant(j.v.x, s0.v.x, c0.v.x, &sn->v.x, &cs->v.x);
        sincos_quadrant(j.v.y, s0.v.y, c0.v.y, &sn->v.y, &cs->v.y);
    }
}

template <typename V, bool FAST>
__device__ __forceinline__ void sincos_t(V x, V* s, V* c) {
    if constexpr (std::is_same<V, double>::value) {
        Real<double>::sincos(x, s, c);
    } else if constexpr (std::is_same<V, float>::value) {
        if constexpr (FAST) { *s = __sinf(x); *c = __cosf(x); }   // MUFU.SIN / MUFU.COS
        else sincos_f32(x, s, c);
    } else {
        if constexpr (FAST) { *s = F2(__sinf(x.v.x), __sinf(x.v.y)); *c = F2(__cosf(x.v.x), __cosf(x.v.y)); }
        else sincos_f32(x, s, c);
    }
}

template <typename V, bool FAST>
__device__ __forceinline__ Trig6<V> trig6(V phi, V theta, V psi) {
    Trig6<V> g;
    sincos_t<V, FAST>(phi, &g.sph, &g.cph);
    sincos_t<V, FAST>(theta, &g.sth, &g.cth);
    sincos_t<V, FAST>(psi, &g.sps, &g.cps);
    return g;
}

// sin / cos of (anchor + d) from the anchor's values by the addition theorem
// with short Taylor polynomials: no range reduction, no quadrant logic, FMA pipe
// only.  Truncation error < 1.3e-8 (sin) / 4e-10 (cos) for |d| <= 0.25, i.e. below
// half an ulp of the result scale.  Used for RK4 stages 2-4, whose angles differ
// from the stage-1 angles by d = c_k * k_angle exactly (fp32 only).
#define MVRL_TRIG_DELTA_MAX2 0.0625f   // (0.25 rad)^2, tested against d_phi^2 + d_theta^2 + d_psi^2
template <typename V>
__device__ __forceinline__ void sincos_delta(V s0, V c0, V d, V z, V* s, V* c) {
    V ps = fmaf_t(z, V(8.333333333e-3f), V(-1.666666667e-1f));
    const V sd = fmaf_t(d * z, ps, d);
    V pc = fmaf_t(z, V(-1.388888889e-3f), V(4.166666667e-2f));
    pc = fmaf_t(z, pc, V(-0.5f));
    const V cd = fmaf_t(z, pc, V(1.0f));
    *s = fmaf_t(s0, cd, c0 * sd);
    *c = fmaf_t(c0, cd, -(s0 * sd));
}

// 6DoF.py:271-275 + 233-236: saturate, deadband, static thrust.
template <typename V, typename S> __device__ __forceinline__ V thruster_force(const Rov6Dev<S>& P, V rpm) {
    V r = tmax(V(-P.rpm_max), tmin(V(P.rpm_max), rpm));
    r = r * vmask_ge(tabs(r), V(P.rpm_db));   // dead band as a 0 / 1 factor (one FSET per lane + a packed multiply)
    return V(P.thrust_k) * r * tabs(r);
}

// H = sum_i F_i A[:, i]  (6DoF.py:278-282).  SP: the reference's default
// allocation pattern - horizontal thrusters 0-3 produce no heave force,
// vertical thrusters 4-7 produce heave, roll and pitch only.
template <typename V, bool SP, typename S>
__device__ __forceinline__ void thrust_wrench(const Rov6Dev<S>& P, const V (&F)[8], V (&H)[6]) {
    if (!P.thrusters_on) {
#pragma unroll
        for (int k = 0; k < 6; ++k) H[k] = V(S(0));
        return;
    }
    auto dot = [&](int k, int lo, int hi) {
        V s = V(P.A[k][lo]) * F[lo];
#pragma unroll
        for (int i = lo + 1; i < hi; ++i) s = fmaf_t(V(P.A[k][i]), F[i], s);
        return s;
    };
    if constexpr (SP) {
        H[0] = dot(0, 0, 4); H[1] = dot(1, 0, 4); H[2] = dot(2, 4, 8);
        H[3] = dot(3, 0, 8); H[4] = dot(4, 0, 8); H[5] = dot(5, 0, 4);
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) H[k] = dot(k, 0, 8);
    }
}

// 6DoF.py:220-231 (+ 238-248): earth-frame demand -> body frame (forces AND
// moments rotated like vectors through the intrinsic-XYZ axes) -> Ainv -> rpm.
// Returns the allocated per-thruster force demand c_i (newtons); rpm_i =
// sign(c_i) sqrt(|c_i| / (rho D^4 Kt)) 60.
template <typename V, bool SP, typename S>
__device__ __forceinline__ void allocate_demand(const Rov6Dev<S>& P, const Trig6<V>& g, const V (&gcf)[6], V (&c)[8]) {
    // body axes of R = Rx(phi) Ry(theta) Rz(psi); every FMA is written out (the translation unit is compiled
    // with -fmad=false so that the one- and two-environment instantiations execute the same operations)
    const V ss = g.sph * g.sth, cs = g.cph * g.sth;
    const V ix = g.cth * g.cps, iy = fmaf_t(ss, g.cps, g.cph * g.sps), iz = fmaf_t(-cs, g.cps, g.sph * g.sps);
    const V jx = -(g.cth * g.sps), jy = fmaf_t(-ss, g.sps, g.cph * g.cps), jz = fmaf_t(cs, g.sps, g.sph * g.cps);
    const V kx = g.sth, ky = -(g.sph * g.cth), kz = g.cph * g.cth;
    V b[6];
    b[0] = fmaf_t(gcf[2], iz, fmaf_t(gcf[1], iy, gcf[0] * ix));
    b[1] = fmaf_t(gcf[2], jz, fmaf_t(gcf[1], jy, gcf[0] * jx));
    b[2] = fmaf_t(gcf[2], kz, fmaf_t(gcf[1], ky, gcf[0] * kx));
    b[3] = fmaf_t(gcf[5], iz, fmaf_t(gcf[4], iy, gcf[3] * ix));
    b[4] = fmaf_t(gcf[5], jz, fmaf_t(gcf[4], jy, gcf[3] * jx));
    b[5] = fmaf_t(gcf[5], kz, fmaf_t(gcf[4], ky, gcf[3] * kx));
    if constexpr (SP) {
        // pinv of the default A: horizontals see (X, Y, N) only, verticals see (Z, K, M) only
#pragma unroll
        for (int i = 0; i < 4; ++i) c[i] = fmaf_t(V(P.Ainv[i][5]), b[5], fmaf_t(V(P.Ainv[i][1]), b[1], V(P.Ainv[i][0]) * b[0]));
#pragma unroll
        for (int i = 4; i < 8; ++i) {
            V s = V(P.Ainv[i][0]) * b[0];
#pragma unroll
            for (int k = 1; k < 5; ++k) s = fmaf_t(V(P.Ainv[i][k]), b[k], s);
            c[i] = s;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            V s = V(P.Ainv[i][0]) * b[0];
#pragma unroll
            for (int k = 1; k < 6; ++k) s = fmaf_t(V(P.Ainv[i][k]), b[k], s);
            c[i] = s;
        }
    }
}

template <typename T> __device__ __forceinline__ T demand_to_rpm(const Rov6Dev<T>& P, T c) {
    return sgn(c) * Real<T>::sqrt(tabs(c) * P.inv_thrust_coef) * T(60);
}

// Thruster force from an allocated demand.  Instead of the reference's literal
// chain (rpm via sqrt, limit, thrust law) the algebraic identity F(rpm(c)) = c
// is used with the limits moved to force space (|c| > F(rpm_max) saturates,
// |c| < F(deadband) is zero): same result up to rounding, no sqrt.
template <typename V, typename S>
__device__ __forceinline__ V demand_to_force(const Rov6Dev<S>& P, V c) {
    // two min / max and one compare per lane (ALU pipe), one packed multiply; the round-1 form (|c|, min, select,
    // copysign) took four ALU instructions per lane and was the largest single consumer of that pipe
    const V sat = tmax(V(-P.f_max), tmin(V(P.f_max), c));
    return sat * vmask_ge(tabs(c), V(P.f_db));
}

// RHS = -Crb v - (Ca + D) v - G + H ; acc = Minv RHS   (6DoF.py:284-396, 428)
// comp (nullable, one-environment types only): -Crb v, -Ca v, -D v, G as in forceModel(retComp=True).
template <typename V, bool SP, typename S>
__device__ __forceinline__ void body_accel(const Rov6Dev<S>& P, const Trig6<V>& g, const V (&nu)[6], const V (&H)[6],
                                           V (&acc)[6], V (&rhs)[6], S* comp = nullptr, long comp_ld = 0) {
    const V u = nu[0], v = nu[1], w = nu[2], p = nu[3], q = nu[4], r = nu[5];
    if constexpr (SP) {
        if (comp == nullptr) {
            // Default sparsity, no component dump: Crb v + Ca v folded analytically (xg = yg = 0,
            // diagonal inertia; the m w v - m v w pairs of 6DoF.py:313-331 cancel identically) and
            // grouped by shared factors:
            //   rhs0 = .. + r (mY v - mzg p) - mZ w q        rhs3 = .. - w (cVW v + mzg p) + r (mzg u - cQR q)
            //   rhs1 = .. - r (mX u + mzg q) + mZ w p        rhs4 = .. - w (cUW u + mzg q) + r (mzg v - cPR p)
            //   rhs2 = .. + q (mX u + mzg q) - p (mY v - mzg p)
            const V zp = V(P.mzg) * p, zq = V(P.mzg) * q, cw = V(P.mZ) * w;
            const V ae = fmaf_t(V(P.mX), u, zq), bd = fmaf_t(V(P.mY), v, -zp);
            rhs[0] = fmaf_t(fmaf_t(V(P.Xuu), tabs(u), V(P.Xu)), u, fmaf_t(r, bd, fmaf_t(-cw, q, H[0])));
            rhs[1] = fmaf_t(fmaf_t(V(P.Yvv), tabs(v), V(P.Yv)), v, fmaf_t(-r, ae, fmaf_t(cw, p, H[1])));
            rhs[2] = fmaf_t(fmaf_t(V(P.Zww), tabs(w), V(P.Zw)), w, fmaf_t(q, ae, fmaf_t(-p, bd, H[2])));
            const V t1 = fmaf_t(V(P.cVW), v, zp), t2 = fmaf_t(V(-P.cQR), q, V(P.mzg) * u);
            const V t3 = fmaf_t(V(P.cUW), u, zq), t4 = fmaf_t(V(-P.cPR), p, V(P.mzg) * v);
            rhs[3] = fmaf_t(fmaf_t(V(P.Kpp), tabs(p), V(P.Kp)), p,
                            fmaf_t(V(-P.gz), g.cth * g.sph, fmaf_t(-w, t1, fmaf_t(r, t2, H[3]))));
            rhs[4] = fmaf_t(fmaf_t(V(P.Mqq), tabs(q), V(P.Mq)), q,
                            fmaf_t(V(P.Mww) * tabs(w), w, fmaf_t(V(-P.gz), g.sth, fmaf_t(-w, t3, fmaf_t(r, t4, H[4])))));
            rhs[5] = fmaf_t(fmaf_t(V(P.Nrr), tabs(r), V(P.Nr)), r, fmaf_t(V(-P.cPQ) * p, q, fmaf_t(V(-P.cUV) * u, v, H[5])));
            acc[0] = fmaf_t(V(P.Minv[0][4]), rhs[4], V(P.Minv[0][0]) * rhs[0]);
            acc[1] = fmaf_t(V(P.Minv[1][3]), rhs[3], V(P.Minv[1][1]) * rhs[1]);
            acc[2] = V(P.Minv[2][2]) * rhs[2];
            acc[3] = fmaf_t(V(P.Minv[3][1]), rhs[1], V(P.Minv[3][3]) * rhs[3]);
            acc[4] = fmaf_t(V(P.Minv[4][0]), rhs[0], V(P.Minv[4][4]) * rhs[4]);
            acc[5] = V(P.Minv[5][5]) * rhs[5];
            return;
        }
    }
    const V m = V(P.m);
    V crb[6], ca[6], dv[6], G[6];

    // ---- Crb(v) v, 6DoF.py:303-332
    if constexpr (SP) {  // xg = yg = 0, diagonal inertia
        const V zr = V(P.zg) * r, zp = V(P.zg) * p, zq = V(P.zg) * q;
        const V a1 = m * zr, b1 = m * w, b2 = m * zr;
        const V c1 = m * (zp - v), c2 = m * (zq + u);
        const V mw = m * w, mv = m * v, mu = m * u;
        crb[0] = a1 * p + mw * q - mv * r;
        crb[1] = -(b1 * p) + b2 * q + mu * r;
        crb[2] = -(c1 * p) - c2 * q;
        const V i1 = V(P.Izz) * r, i2 = -(V(P.Iyy) * q), i3 = V(P.Ixx) * p;
        crb[3] = -(a1 * u) + b1 * v + c1 * w + i1 * q + i2 * r;
        crb[4] = -(mw * u) - b2 * v + c2 * w - i1 * p + i3 * r;
        crb[5] = mv * u - mu * v - i2 * p - i3 * q;
    } else {
        const V a1 = m * (V(P.yg) * q + V(P.zg) * r), a2 = m * (V(P.xg) * q - w), a3 = m * (V(P.xg) * r + v);
        const V b1 = m * (V(P.yg) * p + w), b2 = m * (V(P.zg) * r + V(P.xg) * p), b3 = m * (V(P.yg) * r - u);
        const V c1 = m * (V(P.zg) * p - v), c2 = m * (V(P.zg) * q + u), c3 = m * (V(P.xg) * p + V(P.yg) * q);
        const V i1 = -(V(P.Iyz) * q) - V(P.Ixz) * p + V(P.Izz) * r;
        const V i2 = V(P.Iyz) * r + V(P.Ixy) * p - V(P.Iyy) * q;
        const V i3 = -(V(P.Ixz) * r) - V(P.Ixy) * q + V(P.Ixx) * p;
        crb[0] = a1 * p - a2 * q - a3 * r;
        crb[1] = -(b1 * p) + b2 * q - b3 * r;
        crb[2] = -(c1 * p) - c2 * q + c3 * r;
        crb[3] = -(a1 * u) + b1 * v + c1 * w + i1 * q + i2 * r;
        crb[4] = a2 * u - b2 * v + c2 * w - i1 * p + i3 * r;
        crb[5] = a3 * u + b3 * v - c3 * w - i2 * p - i3 * q;
    }

    // ---- Ca(v) v, 6DoF.py:334-341 (Zwdot here although Ma carries Zvdot)
    {
        const V xu = V(P.Xud) * u, yv = V(P.Yvd) * v, zw = V(P.Zwd) * w, kp = V(P.Kpd) * p, mq = V(P.Mqd) * q, nr = V(P.Nrd) * r;
        ca[0] = -(zw * q) + yv * r;
        ca[1] = zw * p - xu * r;
        ca[2] = -(yv * p) + xu * q;
        ca[3] = -(zw * v) + yv * w - nr * q + mq * r;
        ca[4] = zw * u - xu * w + nr * p - kp * r;
        ca[5] = -(yv * u) + xu * v - mq * p + kp * q;
    }

    // ---- -D(v) v, 6DoF.py:345-370: D = -(Dl + Dq |v|)
    {
        const V au = tabs(u), av = tabs(v), aw = tabs(w), ap = tabs(p), aq = tabs(q), ar = tabs(r);
        dv[0] = (V(P.Xu) + V(P.Xuu) * au) * u;
        if constexpr (SP) {  // only Mww couples
            dv[1] = (V(P.Yv) + V(P.Yvv) * av) * v;
            dv[2] = (V(P.Zw) + V(P.Zww) * aw) * w;
            dv[3] = (V(P.Kp) + V(P.Kpp) * ap) * p;
            dv[4] = (V(P.Mww) * aw) * w + (V(P.Mq) + V(P.Mqq) * aq) * q;
            dv[5] = (V(P.Nr) + V(P.Nrr) * ar) * r;
        } else {
            dv[1] = (V(P.Yv) + V(P.Yvv) * av) * v + (V(P.Yp) + V(P.Ypp) * ap) * p + (V(P.Yr) + V(P.Yrr) * ar) * r;
            dv[2] = (V(P.Zw) + V(P.Zww) * aw) * w + (V(P.Zq) + V(P.Zqq) * aq) * q;
            dv[3] = (V(P.Kv) + V(P.Kvv) * av) * v + (V(P.Kp) + V(P.Kpp) * ap) * p + (V(P.Kr) + V(P.Krr) * ar) * r;
            dv[4] = (V(P.Mw) + V(P.Mww) * aw) * w + (V(P.Mq) + V(P.Mqq) * aq) * q;
            dv[5] = (V(P.Nv) + V(P.Nvv) * av) * v + (V(P.Np) + V(P.Npp) * ap) * p + (V(P.Nr) + V(P.Nrr) * ar) * r;
        }
    }

    // ---- G(phi, theta), 6DoF.py:374-388
    if constexpr (SP) {  // neutrally buoyant, CG/CB on the z axis
        G[0] = V(S(0)); G[1] = V(S(0)); G[2] = V(S(0));
        G[3] = V(P.gz) * g.cth * g.sph;
        G[4] = V(P.gz) * g.sth;
        G[5] = V(S(0));
    } else {
        G[0] = V(P.WmB) * g.sth;
        G[1] = -(V(P.WmB) * g.cth * g.sph);
        G[2] = -(V(P.WmB) * g.cth * g.cph);
        G[3] = -(V(P.gy) * g.cth * g.cph) + V(P.gz) * g.cth * g.sph;
        G[4] = V(P.gz) * g.sth + V(P.gx) * g.cth * g.cph;
        G[5] = -(V(P.gx) * g.cth * g.sph) - V(P.gy) * g.sth;
    }

#pragma unroll
    for (int k = 0; k < 6; ++k) rhs[k] = -crb[k] - ca[k] + dv[k] - G[k] + H[k];

    if constexpr (std::is_same<V, S>::value) {
        if (comp != nullptr) {
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                comp[(0 * 6 + k) * comp_ld] = -crb[k];
                comp[(1 * 6 + k) * comp_ld] = -ca[k];
                comp[(2 * 6 + k) * comp_ld] = dv[k];
                comp[(3 * 6 + k) * comp_ld] = G[k];
                comp[(4 * 6 + k) * comp_ld] = H[k];
            }
        }
    }

    // ---- acc = M^-1 RHS (M is state independent, 6DoF.py:286-299, 428)
    if constexpr (SP) {  // couplings (0,4) and (1,3) only
        acc[0] = V(P.Minv[0][0]) * rhs[0] + V(P.Minv[0][4]) * rhs[4];
        acc[1] = V(P.Minv[1][1]) * rhs[1] + V(P.Minv[1][3]) * rhs[3];
        acc[2] = V(P.Minv[2][2]) * rhs[2];
        acc[3] = V(P.Minv[3][1]) * rhs[1] + V(P.Minv[3][3]) * rhs[3];
        acc[4] = V(P.Minv[4][0]) * rhs[0] + V(P.Minv[4][4]) * rhs[4];
        acc[5] = V(P.Minv[5][5]) * rhs[5];
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            V s = V(S(0));
#pragma unroll
            for (int j = 0; j < 6; ++j) s += V(P.Minv[k][j]) * rhs[j];
            acc[k] = s;
        }
    }
}

// 1 / den for the clamped |den| >= 1e-6 of the kinematics
// The bare MUFU.RCP.  1e-6 <= |den| <= 1 here, so neither the operand nor the result is subnormal and the flush-to-zero
// form returns the same bits as __fdividef(1.0f, den) - which, in a translation unit compiled without -ftz, wraps the
// MUFU in a subnormal-operand rescue (x 2^24, compare, two selects, x scale: 2 FMUL + FSETP + 2 FSEL per lane and RK4
// stage = 40 of the rpm loop's 743 instructions per sub-step, 16 of them on the FMA pipe).
__device__ __forceinline__ float rcp_mufu(float den) {
    float inv;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(inv) : "f"(den));
    return inv;
}
template <bool FAST> __device__ __forceinline__ float recip_clamped(float den) {
    // MUFU.RCP needs no special-case path here; one Newton step brings it to <= 1 ulp in the accurate mode
    float inv = rcp_mufu(den);
    if constexpr (!FAST) inv = fmaf(inv, fmaf(-den, inv, 1.0f), inv);
    return inv;
}
template <bool FAST> __device__ __forceinline__ double recip_clamped(double den) { return 1.0 / den; }
template <bool FAST> __device__ __forceinline__ F2 recip_clamped(F2 den) {
    F2 inv = F2(rcp_mufu(den.v.x), rcp_mufu(den.v.y));
    if constexpr (!FAST) inv = fmaf_t(inv, fmaf_t(-den, inv, F2(1.0f)), inv);
    return inv;
}

// eta_dot = J(phi, theta, psi) v  (resources.py:115-141, 6DoF.py:432-435).
// J1[0][2] keeps the reference's sin(phi) in its second term; cos(theta) in
// J2 is clamped exactly as resources.py:116-120.
template <typename V, bool FAST>
__device__ __forceinline__ void kinematics6(const Trig6<V>& g, const V (&nu)[6], V (&ed)[6]) {
    using S = typename VT<V>::S;
    const V u = nu[0], v = nu[1], w = nu[2], p = nu[3], q = nu[4], r = nu[5];
    // J1 v factored through psi: x' = c(psi) A1 - s(psi) B, y' = s(psi) A2 + c(psi) B with
    // A1 = c(th) u + s(th)s(ph) (v + w)   <- the reference's J1[0][2] (sin(phi), not cos(phi))
    // A2 = c(th) u + s(th)s(ph) v + s(th)c(ph) w,  B = c(ph) v - s(ph) w
    const V ss = g.sth * g.sph, sc = g.sth * g.cph, cu = g.cth * u;
    const V A1 = fmaf_t(ss, v + w, cu);
    const V A2 = fmaf_t(sc, w, fmaf_t(ss, v, cu));
    const V B = fmaf_t(g.cph, v, -(g.sph * w));
    ed[0] = fmaf_t(g.cps, A1, -(g.sps * B));
    ed[1] = fmaf_t(g.sps, A2, g.cps * B);
    ed[2] = fmaf_t(g.cth, fmaf_t(g.sph, v, g.cph * w), -(g.sth * u));
    // resources.py:116-120, branch-free: |c| < 1e-12 -> 1e-6, |c| < 1e-6 -> 1e-6 sign(c)
    const V ad = tabs(g.cth);
    const V tiny = vsel(vlt(ad, V(S(1e-12))), V(S(1e-6)), vcopysign(V(S(1e-6)), g.cth));
    const V den = vsel(vlt(ad, V(S(1e-6))), tiny, g.cth);
    const V inv = recip_clamped<FAST>(den);
    const V a = fmaf_t(g.sph, q, g.cph * r);  // shared by rows 0 and 2 of J2
    ed[5] = inv * a;
    ed[3] = fmaf_t(g.sth, ed[5], p);
    ed[4] = fmaf_t(g.cph, q, -(g.sph * r));
}

// controller error of BlueROV2Heavy6DoF_PID_controller.computeControlForces (6DoF.py:55-61):
// roll / pitch errors are raw differences, only yaw is wrapped
template <typename V> __device__ __forceinline__ void pid6_error(const V (&sp)[6], const V (&pose)[6], V (&e)[6]) {
#pragma unroll
    for (int k = 0; k < 5; ++k) e[k] = sp[k] - pose[k];
    e[5] = angle_error_v(sp[5], pose[5]);
}

// BlueROV2Heavy6DoF_PID_controller.computeControlForces, 6DoF.py:43-73.
// dtc = t - tOld (the same for every environment of a thread).  e_old[0] = NaN encodes eOld is None.
// CHECK_NONE = false: the caller has already replaced a None eOld by the error of the first call (pid6_prime),
// which is what 6DoF.py:62-63 does - saves 13 selects per call inside the RK4 loop of the step kernel.
// inv_dt = 1 / max(1e-9, dtc) and half_dt = dtc / 2 are passed in: the step kernel gets them from the host
// (uniform registers), pid6() below derives them from a per-environment dtc.
template <bool CHECK_NONE = true, typename V, typename S>
__device__ __forceinline__ void pid6_core(const Rov6Dev<S>& P, V (&e_old)[6], V (&e_int)[6], const V (&sp)[6],
                                          const V (&pose)[6], S inv_dt, S half_dt, V (&out)[6]) {
    V e[6];
    pid6_error(sp, pose, e);
    const auto none = visnan(e_old[0]);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const V eo = CHECK_NONE ? vsel(none, e[k], e_old[k]) : e_old[k];
        const V dedt = (e[k] - eo) * V(inv_dt);
        V ei = fmaf_t(V(half_dt), eo + e[k], e_int[k]);
        ei = vsel(vgt(tabs(e[k]), V(P.pWind[k])), V(S(0)), ei);
        const V cvl = fmaf_t(V(P.pKi[k]), ei, fmaf_t(V(P.pKd[k]), dedt, V(P.pKp[k]) * e[k]));
        out[k] = tmax(V(-P.pMax[k]), tmin(V(P.pMax[k]), cvl));
        e_int[k] = ei;
        e_old[k] = e[k];
    }
}

// The same controller for the fp32 step kernels, with e - eOld taken from the pose INCREMENT between two consecutive
// calls instead of from two rounded errors.  Inside an env step the set-point is constant, so e - eOld = -(pose -
// pose_old) exactly, and the step kernel knows that increment as a difference of RK4 offsets c k (a few ulp of the
// INCREMENT), whereas sp - pose carries half an ulp of the POSE.  It matters because RK4 stages 1 and 3 are evaluated
// at the same t as the call before them: dedt = (e - eOld) / 1e-9 (6DoF.py:64) turns the SIGN of a ~1e-4 difference
// into a saturated +-pMax demand, and in fp32 the rounded errors get that sign wrong in ~1e-3 of the calls, the
// increments in ~1e-7 (measured: tests/test_parity_modes_gpu.py).  dpose[k] = pose_k - (pose_k of the previous call);
// the wrapped yaw error may jump by 2 pi between two calls - then the literal difference is used (it is large and
// its sign is not in question).  The caller primes dpose with eOld - e for the first call of an env step, where the
// set-point has moved and the literal difference is the right one.
template <bool INTEGRATE, typename V, typename S>
__device__ __forceinline__ void pid6_core_dp(const Rov6Dev<S>& P, V (&e_old)[6], V (&e_int)[6], const V (&sp)[6],
                                             const V (&pose)[6], const V (&dpose)[6], const S (&kd_inv_dt)[6], S half_dt, V (&out)[6]) {
    V e[6];
    pid6_error(sp, pose, e);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        V de = -dpose[k];
        if (k == 5) {
            const V dd = e[5] - e_old[5];
            de = vsel(vgt(tabs(dd), V(S(1))), dd, de);
        }
        // anti-wind-up (6DoF.py:67) folded into the integrator update as a 0 / 1 factor.  INTEGRATE = false: a call at
        // the same t as the one before it (half_dt = 0) adds nothing to the integral - only the wind-up test applies.
        V ei = e_int[k];
        if constexpr (INTEGRATE) ei = fmaf_t(V(half_dt), e_old[k] + e[k], ei);
        ei = ei * vmask_le(tabs(e[k]), V(P.pWind[k]));
        // Kd dedt = (Kd / max(1e-9, dt)) (e - eOld): the quotient comes from the host (uniform register)
        const V cvl = fmaf_t(V(P.pKi[k]), ei, fmaf_t(V(kd_inv_dt[k]), de, V(P.pKp[k]) * e[k]));
        out[k] = tmax(V(-P.pMax[k]), tmin(V(P.pMax[k]), cvl));
        e_int[k] = ei;
        e_old[k] = e[k];
    }
}

template <typename V, typename S>
__device__ __forceinline__ void pid6(const Rov6Dev<S>& P, V (&e_old)[6], V (&e_int)[6], const V (&sp)[6],
                                     const V (&pose)[6], S dtc, V (&out)[6]) {
    pid6_core<true>(P, e_old, e_int, sp, pose, S(1) / tmax(S(1e-9), dtc), S(0.5) * dtc, out);
}

// eOld of a fresh controller := the error its first call will see (pose = the state at the start of the env step)
template <typename V> __device__ __forceinline__ void pid6_prime(V (&e_old)[6], const V (&sp)[6], const V (&pose)[6]) {
    const auto none = visnan(e_old[0]);
    if (vany(none)) {
        V e[6];
        pid6_error(sp, pose, e);
#pragma unroll
        for (int k = 0; k < 6; ++k) e_old[k] = vsel(none, e[k], e_old[k]);
    }
}

}  // namespace mvrl
