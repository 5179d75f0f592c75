// BlueROV2 Heavy 3DoF (surge / sway / yaw) model and env step, K3.
// Restates dynamicsModel_BlueROV2_Heavy_3DoF.py:114-296 (model, built-in PID,
// jet-drag thruster augment) and :397-514 (env).  One environment per thread.
#pragma once
#include "mvrl_math.cuh"
#include "rov6_kernels.cuh"  // stats_accumulate, ACT_* enums

namespace mvrl {

template <typename T> struct Rov3Dev {
    T m, xg, yg;
    T Xud, Yvd;
    T Xu, Yv, Yr, Nv, Nr, Xuu, Yvv, Yrr, Nvv, Nrr;
    T Minv[3][3];
    T Ainv[4][3];
    T thrust_k, inv_thrust_coef, rpm_max, rpm_db;
    T inv_jet_area;   // 1 / (0.5 rho pi D^2)           (3DoF.py:121)
    T drag_k;         // -0.5 rho dispVol^(2/3)           (3DoF.py:124)
    T cos_a, sin_a, arm;  // thruster angle, sqrt(l_x^2 + l_y^2) (3DoF.py:256-263)
    T pKp[3], pKi[3], pKd[3], pWind[3], pMax[3];
    T inv_3L, act_pos, act_ang, inv_ang;
};

// 3DoF.py:114-126
template <typename T>
__device__ __forceinline__ void thruster_model3(const Rov3Dev<T>& P, T u, T rpm, T* F, T* X) {
    const T f = P.thrust_k * rpm * tabs(rpm);
    const T u_jet = Real<T>::sqrt(tabs(f) * P.inv_jet_area);
    const T q = tabs(u) / tmax(T(1e-5), u_jet);
    const T dcd = T(0.56599) * Real<T>::exp(T(-7.60891) * q) + T(0.05654) * Real<T>::exp(T(-0.89679) * q);
    *F = f;
    *X = dcd * P.drag_k * tabs(u) * u;
}

template <typename T> __device__ __forceinline__ T limit_rpm3(const Rov3Dev<T>& P, T rpm) {  // 3DoF.py:171-175
    T r = tmax(-P.rpm_max, tmin(P.rpm_max, rpm));
    return tabs(r) < P.rpm_db ? T(0) : r;
}

// 3DoF.py:141-157
template <typename T>
__device__ __forceinline__ void pid3(const Rov3Dev<T>& P, T (&e_old)[3], T (&e_int)[3], const T (&sp)[3], T x, T y, T psi, T dtc, T (&out)[3]) {
    T e[3] = {sp[0] - x, sp[1] - y, angle_error(sp[2], psi)};
    const bool none = e_old[0] != e_old[0];
    const T inv_dt = T(1) / tmax(T(1e-9), dtc);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const T eo = none ? e[k] : e_old[k];
        const T dedt = (e[k] - eo) * inv_dt;
        T ei = e_int[k] + T(0.5) * (eo + e[k]) * dtc;
        if (tabs(e[k]) > P.pWind[k]) ei = T(0);
        const T c = P.pKp[k] * e[k] + P.pKd[k] * dedt + P.pKi[k] * ei;
        out[k] = tmax(-P.pMax[k], tmin(P.pMax[k], c));
        e_int[k] = ei;
        e_old[k] = e[k];
    }
}

// The fp32 step kernel's variant: e - eOld from the pose increment between two consecutive calls (see pid6_core_dp in
// rov6_model.cuh for the why); dpose[k] = pose_k - pose_k of the previous call, primed with eOld - e for the first call
// of an env step.  A 2 pi jump of the wrapped yaw error falls back to the literal difference.
template <typename T>
__device__ __forceinline__ void pid3_dp(const Rov3Dev<T>& P, T (&e_old)[3], T (&e_int)[3], const T (&sp)[3], T x, T y, T psi,
                                        const T (&dpose)[3], T dtc, T (&out)[3]) {
    T e[3] = {sp[0] - x, sp[1] - y, angle_error(sp[2], psi)};
    const T inv_dt = T(1) / tmax(T(1e-9), dtc);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        T de = -dpose[k];
        if (k == 2) { const T dd = e[2] - e_old[2]; if (tabs(dd) > T(1)) de = dd; }
        const T dedt = de * inv_dt;
        T ei = e_int[k] + T(0.5) * (e_old[k] + e[k]) * dtc;
        if (tabs(e[k]) > P.pWind[k]) ei = T(0);
        const T c = P.pKp[k] * e[k] + P.pKd[k] * dedt + P.pKi[k] * ei;
        out[k] = tmax(-P.pMax[k], tmin(P.pMax[k], c));
        e_int[k] = ei;
        e_old[k] = e[k];
    }
}

// 3DoF.py:159-168: earth-frame PID output -> body frame -> rpm
template <typename T>
__device__ __forceinline__ void allocate3(const Rov3Dev<T>& P, T s, T c, const T (&cvl)[3], T (&gcf)[3], T (&rpm)[4]) {
    gcf[0] = cvl[0] * c + cvl[1] * s;
    gcf[1] = -cvl[0] * s + cvl[1] * c;
    gcf[2] = cvl[2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const T d = P.Ainv[i][0] * gcf[0] + P.Ainv[i][1] * gcf[1] + P.Ainv[i][2] * gcf[2];
        rpm[i] = sgn(d) * Real<T>::sqrt(tabs(d) * P.inv_thrust_coef) * T(60);
    }
}

// 3DoF.py:170-296 from the limited rpm on.  s = [x, y, psi, u, v, r].
template <typename T>
__device__ __forceinline__ void derivs3_core(const Rov3Dev<T>& P, T sps, T cps, T u, T v, T r, const T (&rpm)[4], T (&k)[6]) {
    T F[4], X[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) thruster_model3(P, u, limit_rpm3(P, rpm[i]), &F[i], &X[i]);
    const T Xh = X[0] + X[1] + X[2] + X[3] + (F[0] + F[1] - F[2] - F[3]) * P.cos_a;
    const T Yh = (F[0] - F[1] + F[2] - F[3]) * P.sin_a;
    const T Nh = P.arm * (F[0] + F[1] + F[2] + F[3]);
    const T m = P.m;
    const T c13 = -m * (P.xg * r + v), c23 = -m * (P.yg * r - u);
    const T crb0 = c13 * r, crb1 = c23 * r, crb2 = -c13 * u - c23 * v;
    const T ca0 = P.Yvd * v * r, ca1 = -P.Xud * u * r, ca2 = -P.Yvd * v * u + P.Xud * u * v;
    const T d0 = -(P.Xu + P.Xuu * tabs(u)) * u;
    const T d1 = -((P.Yv + P.Yvv * tabs(v)) * v + (P.Yr + P.Yrr * tabs(r)) * r);
    const T d2 = -((P.Nv + P.Nvv * tabs(v)) * v + (P.Nr + P.Nrr * tabs(r)) * r);
    const T rhs0 = -crb0 - (ca0 + d0) + Xh, rhs1 = -crb1 - (ca1 + d1) + Yh, rhs2 = -crb2 - (ca2 + d2) + Nh;
    k[0] = cps * u - sps * v;
    k[1] = sps * u + cps * v;
    k[2] = r;
#pragma unroll
    for (int i = 0; i < 3; ++i) k[3 + i] = P.Minv[i][0] * rhs0 + P.Minv[i][1] * rhs1 + P.Minv[i][2] * rhs2;
}

// ---------------------------------------------------------------------------
template <typename T> struct Rov3StepArgs {
    Rov3Dev<T> P;
    long n, ld;
    T* state; const T* action; T* obs; T* reward; uint8_t* done; int32_t* istep;
    T* setpoint; T* path; T* ctrl; uint32_t* episode; T* term_obs; T* aux; double* stats;
    T dt, h, hh, h6, h3;   // host-computed step sizes (uniform-register operands, see Rov6StepArgs)
    int n_sub, max_steps;
    unsigned long long seed, env_id0;
    int auto_reset, fixed_sp;
};

// 3DoF.py:397-409
template <typename T>
__device__ __forceinline__ void observe3(const Rov3Dev<T>& P, const T (&y)[6], const T (&path)[4], T sp_psi, T (&obs)[5]) {
    obs[0] = clampt((path[0] - y[0]) * P.inv_3L, T(-1), T(1));
    obs[1] = clampt((path[1] - y[1]) * P.inv_3L, T(-1), T(1));
    obs[2] = clampt((path[2] - y[0]) * P.inv_3L, T(-1), T(1));
    obs[3] = clampt((path[3] - y[1]) * P.inv_3L, T(-1), T(1));
    obs[4] = clampt(angle_error(sp_psi, y[2]) * P.inv_ang, T(-1), T(1));
}

// 3DoF.py:423-424 with Philox instead of the global numpy RNG
template <typename T>
__device__ __forceinline__ void draw_reset3(unsigned long long seed, unsigned long long env, uint32_t episode, T (&path)[4], T* heading) {
    const uint4 a = Philox::draw(seed, env, episode, 0u, 0u);
    const uint4 b = Philox::draw(seed, env, episode, 0u, 1u);
    path[0] = (u01<T>(a.x) - T(0.5)) * T(10); path[1] = (u01<T>(a.y) - T(0.5)) * T(10);
    path[2] = (u01<T>(a.z) - T(0.5)) * T(10); path[3] = (u01<T>(a.w) - T(0.5)) * T(10);
    *heading = u01<T>(b.x) * T(MVRL_TWO_PI);
}

// K3 step: MODE = ACT_RPM (4 rpm, stateless; build addition) or ACT_SETPOINT (3DoF.py:455-514)
template <typename T, int MODE, bool FAST>
__global__ void __launch_bounds__(128)
rov3_step_kernel(const __grid_constant__ Rov3StepArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const Rov3Dev<T>& P = a.P;
    const long ld = a.ld;
    T y[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) y[k] = a.state[k * ld + i];
    const int istep = a.istep[i] + 1;
    constexpr int NA = (MODE == ACT_RPM) ? 4 : 3;
    T act[NA];
#pragma unroll
    for (int k = 0; k < NA; ++k) act[k] = a.action[k * ld + i];
    T sp[3], e_old[3], e_int[3];
    if constexpr (MODE == ACT_SETPOINT) {
        if (a.fixed_sp) {
#pragma unroll
            for (int k = 0; k < 3; ++k) sp[k] = a.setpoint[k * ld + i];
        } else {  // 3DoF.py:469-472
            sp[0] = act[0] * P.act_pos + y[0];
            sp[1] = act[1] * P.act_pos + y[1];
            sp[2] = act[2] * P.act_ang + y[2];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) { e_old[k] = a.ctrl[k * ld + i]; e_int[k] = a.ctrl[(3 + k) * ld + i]; }
    } else {
        sp[2] = a.setpoint[2 * ld + i];
    }
    T path[4];   // epilogue input, loaded early so the latency hides behind the RK4 loop
#pragma unroll
    for (int k = 0; k < 4; ++k) path[k] = a.path[k * ld + i];
    T gcf[3] = {T(0), T(0), T(0)};
    T rpm[4];
    if constexpr (MODE == ACT_RPM) {
#pragma unroll
        for (int k = 0; k < 4; ++k) rpm[k] = act[k];
    }
    // RK4 as in rov6_step_kernel: fp32 pose advanced by the summed increment with a Kahan carry
    constexpr bool COMP = (sizeof(T) == 4) && !FAST && (MVRL_POSE_COMP != 0);
    constexpr bool DPOSE = (MODE == ACT_SETPOINT) && COMP && (MVRL_PID_DPOSE != 0);
    T dpose[3] = {T(0), T(0), T(0)}, off[3] = {T(0), T(0), T(0)};
    if constexpr (DPOSE) {   // first call of the env step: literal e - eOld (a fresh controller has eOld = e)
        const T e0[3] = {sp[0] - y[0], sp[1] - y[1], angle_error(sp[2], y[2])};
        if (e_old[0] != e_old[0]) {
#pragma unroll
            for (int k = 0; k < 3; ++k) e_old[k] = e0[k];
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) dpose[k] = e_old[k] - e0[k];
    }
    auto f = [&](const T (&s)[6], T (&k)[6], T dtc) {
        T sn, cs;
        sincos_t<T, FAST>(s[2], &sn, &cs);
        if constexpr (MODE == ACT_SETPOINT) {
            T cvl[3];
            if constexpr (DPOSE) pid3_dp(P, e_old, e_int, sp, s[0], s[1], s[2], dpose, dtc, cvl);
            else pid3(P, e_old, e_int, sp, s[0], s[1], s[2], dtc, cvl);
            allocate3(P, sn, cs, cvl, gcf, rpm);
        }
        derivs3_core(P, sn, cs, s[3], s[4], s[5], rpm, k);
    };
    const T h = a.h, hh = a.hh, h6 = a.h6, h3 = a.h3;
    T carry[3] = {T(0), T(0), T(0)};
    for (int sub = 0; sub < a.n_sub; ++sub) {
        T k[6], acc[6], yt[6];
#pragma unroll
        for (int j = 0; j < 6; ++j) { acc[j] = (COMP && j < 3) ? T(0) : y[j]; yt[j] = y[j]; }
#pragma unroll
        for (int st = 0; st < 4; ++st) {
            f(yt, k, (st & 1) ? hh : T(0));
            const T wk = (st == 0 || st == 3) ? h6 : h3;
            const T ck = (st == 2) ? h : hh;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                acc[j] = fmaf_t(wk, k[j], acc[j]);
                if (DPOSE && j < 3) {
                    const T o = (st < 3) ? ck * k[j] : acc[j];   // offset of the next call's pose from y
                    dpose[j] = o - off[j];
                    off[j] = (st < 3) ? o : T(0);
                    if (st < 3) yt[j] = y[j] + o;
                } else if (st < 3) {
                    yt[j] = fmaf_t(ck, k[j], y[j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            if (COMP && j < 3) rk4_pose_update(y[j], carry[j], acc[j]);
            else y[j] = acc[j];
        }
    }
    // outside the exact range of the fp32 sin/cos reduction: flagged like rov6_step_kernel, on the yaw at the end of the step
    bool bad = (sizeof(T) == 4) && !FAST && tabs(y[2]) > T(MVRL_SINCOS_F32_MAX_ARG);
    y[2] = pymod_pos(y[2], T(MVRL_TWO_PI));  // 3DoF.py:480
#pragma unroll
    for (int k = 0; k < 6; ++k) bad = bad || !finite_t(y[k]);
    T obs[5];
    observe3(P, y, path, sp[2], obs);
    const bool is_done = istep >= a.max_steps;
    if (a.aux != nullptr) {  // generalisedControlForces(3) + controlVector(4), 3DoF.py:498-500
#pragma unroll
        for (int k = 0; k < 3; ++k) a.aux[k * ld + i] = gcf[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) a.aux[(3 + k) * ld + i] = rpm[k];
    }
    if (a.stats != nullptr) stats_accumulate<false>(a.stats, is_done && a.auto_reset, (double)istep, 0.0, bad);
    int istep_out = istep;
    if (is_done && a.auto_reset) {
        if (a.term_obs != nullptr) {
#pragma unroll
            for (int k = 0; k < 5; ++k) a.term_obs[k * ld + i] = obs[k];
        }
        const uint32_t ep = a.episode[i] + 1u;
        a.episode[i] = ep;
        istep_out = 0;
#pragma unroll
        for (int k = 0; k < 6; ++k) y[k] = T(0);
        if (!a.fixed_sp) {
            T heading;
            draw_reset3<T>(a.seed, a.env_id0 + (unsigned long long)i, ep, path, &heading);
#pragma unroll
            for (int k = 0; k < 4; ++k) a.path[k * ld + i] = path[k];
            sp[0] = path[0]; sp[1] = path[1]; sp[2] = heading;
#pragma unroll
            for (int k = 0; k < 3; ++k) a.setpoint[k * ld + i] = sp[k];
        }
        if constexpr (MODE == ACT_SETPOINT) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { e_old[k] = T(0); e_int[k] = T(0); }
            e_old[0] = Real<T>::nan();
        }
        observe3(P, y, path, sp[2], obs);
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) a.state[k * ld + i] = y[k];
#pragma unroll
    for (int k = 0; k < 5; ++k) a.obs[k * ld + i] = obs[k];
    a.reward[i] = T(0);  // 3DoF.py:495
    a.done[i] = is_done ? 1 : 0;
    a.istep[i] = istep_out;
    if constexpr (MODE == ACT_SETPOINT) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            a.setpoint[k * ld + i] = sp[k];
            a.ctrl[k * ld + i] = e_old[k];
            a.ctrl[(3 + k) * ld + i] = e_int[k];
        }
        a.ctrl[6 * ld + i] = T(istep_out) * a.dt;
    }
}

// K3 derivs (parity entry): MODE RPM: act = rpm[4]; SETPOINT: t, setpoint, ctrl [7][ld]
template <typename T> struct Rov3DerivArgs {
    Rov3Dev<T> P;
    long n, ld;
    const T* state; const T* act; const T* t; const T* setpoint; T* ctrl; T* dstate; T* aux;
};

template <typename T, int MODE>
__global__ void __launch_bounds__(128)
rov3_derivs_kernel(const __grid_constant__ Rov3DerivArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const long ld = a.ld;
    T s[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) s[k] = a.state[k * ld + i];
    T sn, cs;
    Real<T>::sincos(s[2], &sn, &cs);
    T gcf[3] = {T(0), T(0), T(0)}, rpm[4];
    if constexpr (MODE == ACT_RPM) {
#pragma unroll
        for (int k = 0; k < 4; ++k) rpm[k] = a.act[k * ld + i];
    } else {
        T e_old[3], e_int[3], sp[3], cvl[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) { e_old[k] = a.ctrl[k * ld + i]; e_int[k] = a.ctrl[(3 + k) * ld + i]; sp[k] = a.setpoint[k * ld + i]; }
        const T t = a.t[i];
        pid3(a.P, e_old, e_int, sp, s[0], s[1], s[2], t - a.ctrl[6 * ld + i], cvl);
#pragma unroll
        for (int k = 0; k < 3; ++k) { a.ctrl[k * ld + i] = e_old[k]; a.ctrl[(3 + k) * ld + i] = e_int[k]; }
        a.ctrl[6 * ld + i] = t;
        allocate3(a.P, sn, cs, cvl, gcf, rpm);
    }
    T k[6];
    derivs3_core(a.P, sn, cs, s[3], s[4], s[5], rpm, k);
#pragma unroll
    for (int j = 0; j < 6; ++j) a.dstate[j * ld + i] = k[j];
    if (a.aux != nullptr) {
#pragma unroll
        for (int j = 0; j < 3; ++j) a.aux[j * ld + i] = gcf[j];
#pragma unroll
        for (int j = 0; j < 4; ++j) a.aux[(3 + j) * ld + i] = rpm[j];
    }
}

template <typename T> struct Rov3ResetArgs {
    Rov3Dev<T> P;
    long n, ld;
    T* state; T* obs; int32_t* istep; T* setpoint; T* path; T* ctrl; const uint32_t* episode; T* aux;
    const uint8_t* mask;
    T init_sp[3];
    int has_init_sp;
    unsigned long long seed, env_id0;
};

// 3DoF.py:411-453
template <typename T>
__global__ void __launch_bounds__(128)
rov3_reset_kernel(const __grid_constant__ Rov3ResetArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if (a.mask != nullptr && a.mask[i] == 0) return;
    const long ld = a.ld;
    T y[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) { y[k] = T(0); a.state[k * ld + i] = T(0); }
    a.istep[i] = 0;
    T path[4], sp[3];
    if (a.has_init_sp) {
#pragma unroll
        for (int k = 0; k < 3; ++k) sp[k] = a.init_sp[k];
        path[0] = sp[0]; path[1] = sp[1]; path[2] = sp[0]; path[3] = sp[1];
    } else {
        T heading;
        draw_reset3<T>(a.seed, a.env_id0 + (unsigned long long)i, a.episode ? a.episode[i] : 0u, path, &heading);
        sp[0] = path[0]; sp[1] = path[1]; sp[2] = heading;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) a.path[k * ld + i] = path[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) a.setpoint[k * ld + i] = sp[k];
    if (a.ctrl != nullptr) {
#pragma unroll
        for (int k = 0; k < 7; ++k) a.ctrl[k * ld + i] = T(0);
        a.ctrl[i] = Real<T>::nan();
    }
    if (a.aux != nullptr) {
#pragma unroll
        for (int k = 0; k < 7; ++k) a.aux[k * ld + i] = T(0);
    }
    T obs[5];
    observe3(a.P, y, path, sp[2], obs);
#pragma unroll
    for (int k = 0; k < 5; ++k) a.obs[k * ld + i] = obs[k];
}

// ---------------------------------------------------------------------------
// lineOfSight + LOSNavigation.predict (3DoF.py:517-607): the heuristic agent that turns the 5
// observations of the 3DoF env into its 3 actions.  Branch order and NaN behaviour as upstream.
// ---------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void line_of_sight(T p0x, T p0y, T p1x, T p1y, T rnav, T* tx, T* ty) {
    const T d_to_wp = Real<T>::sqrt(p1x * p1x + p1y * p1y);
    if (d_to_wp < rnav) { *tx = p1x; *ty = p1y; return; }
    const T vx = p1x - p0x, vy = p1y - p0y;
    const T d_seg = Real<T>::sqrt(vx * vx + vy * vy);
    const T hx = vx / d_seg, hy = vy / d_seg;
    const T det = p0x * p1y - p1x * p0y;
    const T delta = rnav * rnav * (d_seg * d_seg) - det * det;
    if (delta < T(0)) {  // the segment is out of sight: head for the nearest point of it
        const T d_along = (-p0x) * hx + (-p0y) * hy;
        if (d_along > d_seg) { *tx = p1x; *ty = p1y; }
        else if (d_along < T(0)) { *tx = p0x; *ty = p0y; }
        else { *tx = p0x + d_along * hx; *ty = p0y + d_along * hy; }
        return;
    }
    if (!(delta >= T(0))) { *tx = Real<T>::nan(); *ty = Real<T>::nan(); return; }  // NaN input (upstream: unbound variable)
    T sy = sgn(vy);
    if (tabs(sy) < T(1e-12)) sy = T(1);
    const T lim = tmax(T(1e-6), d_seg);
    const T den = lim * lim, sq = Real<T>::sqrt(delta);
    const T a0x = (det * vy + sy * vx * sq) / den, a0y = (-det * vx + tabs(vy) * sq) / den;
    const T a1x = (det * vy - sy * vx * sq) / den, a1y = (-det * vx - tabs(vy) * sq) / den;
    const T s0 = (hx * (a0x - p0x) + hy * (a0y - p0y)) / lim;
    const T s1 = (hx * (a1x - p0x) + hy * (a1y - p0y)) / lim;
    if (s0 >= T(0) && s0 <= T(1) && s0 > s1) { *tx = a0x; *ty = a0y; }
    else if (s1 >= T(0) && s1 <= T(1)) { *tx = a1x; *ty = a1y; }
    else if (d_to_wp < Real<T>::sqrt(p0x * p0x + p0y * p0y)) { *tx = p1x; *ty = p1y; }
    else { *tx = p0x; *ty = p0y; }
}

// obs T [5][ld] -> action T [3][ld]
template <typename T>
__global__ void los_navigation_kernel(long n, long ld, const T* obs, T* action, T rnav) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T tx, ty;
    line_of_sight(obs[i], obs[ld + i], obs[2 * ld + i], obs[3 * ld + i], rnav, &tx, &ty);
    action[i] = tx; action[ld + i] = ty; action[2 * ld + i] = obs[4 * ld + i];
}

template <typename T>
__global__ void rov3_thruster_kernel(const Rov3Dev<T> P, long n, const T* u, const T* rpm, T* F, T* X) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) thruster_model3(P, u[i], rpm[i], &F[i], &X[i]);
}

}  // namespace mvrl
