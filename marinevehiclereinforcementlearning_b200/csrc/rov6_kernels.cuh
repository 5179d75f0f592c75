// Kernels of the 6DoF path: K1 rov6_step (fused env step), K2 rov6_derivs
// (parity/debug entry), reset and stand-alone PID.  One environment per
// thread; SoA global layout [field][ld] so that every warp-level load/store is
// one fully coalesced 128 B (fp32) / 256 B (fp64) transaction.
#pragma once
#include "rov6_model.cuh"
#include "rov6_default_consts.h"   // generated: the default vehicle's constants as exact float literals (tools/gen_default_consts.py)

namespace mvrl {

enum { ACT_RPM = 0, ACT_FORCE = 1, ACT_SETPOINT = 2 };

template <typename T> struct Rov6StepArgs {
    Rov6Dev<T> P;
    long n, ld;
    T* state; const T* action; T* obs; T* reward; uint8_t* done; int32_t* istep;
    T* setpoint; T* path; T* ctrl; uint32_t* episode; T* term_obs; T* aux; double* stats;
    T pid_inv_dt[2], pid_half_dt[2];   // 1 / max(1e-9, dtc) and dtc / 2 of the PID for dtc = 0 and dtc = h/2 (host-computed, see h6)
    T pid_kd_inv_dt[2][6];             // Kd[k] * pid_inv_dt[half]: derivative gain per unit of e - eOld (fp32 set-point kernels)
    T dt, h, hh, h6, h3;   // env step, RK4 step h = dt / n_sub and h/2, h/6, h/3 - computed on the host: kernel arguments reach the
                           // FMAs through uniform registers, whereas a value computed in the kernel occupies a vector register and
                           // makes every y + c k update an FMA with three register sources (3 instead of 2 pipe cycles as FFMA2)
    int n_sub, max_steps;
    unsigned long long seed, env_id0;
    int auto_reset, fixed_sp;
};

// dataToState, 6DoF.py:467-483 (iWp is always 0 in the reference)
template <typename T>
__device__ __forceinline__ void observe6(const Rov6Dev<T>& P, const T (&y)[12], const T (&path)[6], const T (&sp_ang)[3], T (&obs)[9]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        obs[k] = clampt((path[k] - y[k]) * P.inv_3L, T(-1), T(1));
        obs[3 + k] = clampt((path[3 + k] - y[k]) * P.inv_3L, T(-1), T(1));
        obs[6 + k] = clampt(angle_error(sp_ang[k], y[3 + k]) * P.inv_ang, T(-1), T(1));
    }
}

// 6DoF.py:560 + 467-483 on the fast path: wraps the three angles and fills the observation assuming every
// angle is inside (-2 pi, 4 pi) and every angle error inside (-2 pi, 2 pi); returns false when that does not
// hold (the caller then redoes the angle part with the exact, out-of-line functions).  One test at the end
// instead of a branch per modulo.
// pos[6] = (path - position) / (3 Length) comes in already scaled (the packed kernel forms it for both of a thread's
// environments at once with two packed instructions per way-point component)
template <typename T>
__device__ __forceinline__ bool wrap_observe6_fast(const Rov6Dev<T>& P, const T (&y)[12], const T (&pos)[6], const T (&sp_ang)[3],
                                                   T (&wrapped)[3], T (&obs)[9]) {
    const T tp = T(MVRL_TWO_PI);
    T lo = y[3], hi = y[3], worst = T(0);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        lo = tmin(lo, y[3 + k]); hi = tmax(hi, y[3 + k]);
        wrapped[k] = pymod_small_sel(y[3 + k], tp);
        const T d = sp_ang[k] - wrapped[k];
        worst = tmax(worst, tabs(d));
        obs[k] = clampt(pos[k], T(-1), T(1));
        obs[3 + k] = clampt(pos[3 + k], T(-1), T(1));
        obs[6 + k] = clampt(angle_error_small(d) * P.inv_ang, T(-1), T(1));
    }
    return lo > -tp && hi < tp + tp && worst < tp;   // all false for NaN: the exact path then propagates it
}

// the exact angle part (any magnitude), out of line: wrapped angle and clipped, scaled angle error
template <typename T> struct WrapObs { T wrapped, obs; };   // returned by value: stays in registers
template <typename T>
__device__ __noinline__ WrapObs<T> wrap_angle_exact(T inv_ang, T angle, T sp_angle) {
    WrapObs<T> r;
    r.wrapped = pymod_pos(angle, T(MVRL_TWO_PI));
    r.obs = clampt(angle_error(sp_angle, r.wrapped) * inv_ang, T(-1), T(1));
    return r;
}

// Random branch of reset().  The reference's own line raises (6DoF.py:497,
// shapes (2,3)-(2,)); defined here as the 3-component analogue of 3DoF.py:423:
// path = (U^(2x3) - 0.5) * 10, targetOrientation = U^3 * 2 pi.  Out of line: taken by one
// environment in max_steps, and three Philox blocks would bloat the common path.
template <typename T> struct Reset6 { T path[6]; T orient[3]; };
template <typename T>
__device__ __noinline__ Reset6<T> draw_reset6(unsigned long long seed, unsigned long long env, uint32_t episode) {
    const uint4 a = Philox::draw(seed, env, episode, 0u, 0u);
    const uint4 b = Philox::draw(seed, env, episode, 0u, 1u);
    const uint4 c = Philox::draw(seed, env, episode, 0u, 2u);
    Reset6<T> r;
    r.path[0] = (u01<T>(a.x) - T(0.5)) * T(10); r.path[1] = (u01<T>(a.y) - T(0.5)) * T(10);
    r.path[2] = (u01<T>(a.z) - T(0.5)) * T(10); r.path[3] = (u01<T>(a.w) - T(0.5)) * T(10);
    r.path[4] = (u01<T>(b.x) - T(0.5)) * T(10); r.path[5] = (u01<T>(b.y) - T(0.5)) * T(10);
    r.orient[0] = u01<T>(b.z) * T(MVRL_TWO_PI); r.orient[1] = u01<T>(b.w) * T(MVRL_TWO_PI);
    r.orient[2] = u01<T>(c.x) * T(MVRL_TWO_PI);
    return r;
}

// episode statistics: [episodes, sum length, sum return, min return, max return, non-finite, -, -]
// WITH_RET = false: the env's reward is identically zero (3DoF / 6DoF), so the return statistics are
// the constants 0 - written by plain stores (every writer stores the same value) instead of CAS loops.
template <bool WITH_RET = true>
__device__ __forceinline__ void stats_accumulate(double* stats, bool is_done, double len, double ret, bool bad) {
    const unsigned active = __activemask();
    const unsigned dm = __ballot_sync(active, is_done);
    const unsigned bm = __ballot_sync(active, bad);
    if (dm == 0u && bm == 0u) return;
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(active) - 1;
    if (dm) {
        const double sl = warp_sum(is_done ? len : 0.0, active);
        if constexpr (WITH_RET) {
            const double sr = warp_sum(is_done ? ret : 0.0, active);
            const double mn = warp_min(is_done ? ret : 1.0e300, active);
            const double mx = warp_max(is_done ? ret : -1.0e300, active);
            if (lane == leader) {
                atomicAdd(stats + 0, (double)__popc(dm));
                atomicAdd(stats + 1, sl);
                atomicAdd(stats + 2, sr);
                atomic_min_double(stats + 3, mn);
                atomic_max_double(stats + 4, mx);
            }
        } else if (lane == leader) {
            atomicAdd(stats + 0, (double)__popc(dm));
            atomicAdd(stats + 1, sl);
            stats[3] = 0.0;
            stats[4] = 0.0;
        }
    }
    if (bm && lane == leader) atomicAdd(stats + 5, (double)__popc(bm));
}

// Zero-reward envs (3DoF / 6DoF), counts only: one vote + three hardware warp reductions (REDUX) per thread,
// atomics from one lane of the warps that actually saw a terminal / non-finite environment.
__device__ __forceinline__ void stats_accumulate_counts(double* stats, int n_done, int len_sum, int n_bad) {
    const unsigned active = __activemask();
    if (!__any_sync(active, (n_done | n_bad) != 0)) return;
    const int d = __reduce_add_sync(active, n_done), l = __reduce_add_sync(active, len_sum), b = __reduce_add_sync(active, n_bad);
    if ((int)(threadIdx.x & 31) == __ffs(active) - 1) {
        if (d) {
            atomicAdd(stats + 0, (double)d);
            atomicAdd(stats + 1, (double)l);
            stats[3] = 0.0;   // min / max return: every writer stores the same constant
            stats[4] = 0.0;
        }
        if (b) atomicAdd(stats + 5, (double)b);
    }
}

// Auto-reset of ONE terminated environment (SB3 VecEnv convention; reset semantics of 6DoF.py:485-529), run by
// the step kernel after its regular stores: keeps the terminal observation, bumps the episode counter, zeroes
// the state, draws the next path / target orientation (unless the set-point is fixed), installs a fresh
// controller and writes the observation of the fresh state.  Out of line: one environment in max_steps takes it.
// ep_prev: the environment's episode counter before this reset (the step kernel stages it with the other epilogue inputs)
template <typename T, int MODE>
__device__ __noinline__ void rov6_auto_reset_env(const Rov6StepArgs<T>& a, long i, uint32_t ep_prev) {
    const long ld = a.ld;
    const Rov6Dev<T>& P = a.P;
    if (a.term_obs != nullptr) {
#pragma unroll
        for (int k = 0; k < 9; ++k) a.term_obs[k * ld + i] = a.obs[k * ld + i];
    }
    const uint32_t ep = ep_prev + 1u;
    a.episode[i] = ep;
    a.istep[i] = 0;
#pragma unroll
    for (int k = 0; k < 12; ++k) a.state[k * ld + i] = T(0);
    T path[6], ang[3];
    if (!a.fixed_sp) {
        const Reset6<T> rs = draw_reset6<T>(a.seed, a.env_id0 + (unsigned long long)i, ep);
#pragma unroll
        for (int k = 0; k < 6; ++k) { path[k] = rs.path[k]; a.path[k * ld + i] = path[k]; }
#pragma unroll
        for (int k = 0; k < 3; ++k) { ang[k] = rs.orient[k]; a.setpoint[k * ld + i] = path[k]; a.setpoint[(3 + k) * ld + i] = ang[k]; }
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) path[k] = a.path[k * ld + i];
#pragma unroll
        for (int k = 0; k < 3; ++k) ang[k] = a.setpoint[(3 + k) * ld + i];
    }
    if constexpr (MODE == ACT_SETPOINT) {  // fresh controller, 6DoF.py:37-41, 514
#pragma unroll
        for (int k = 0; k < 13; ++k) a.ctrl[k * ld + i] = T(0);
        a.ctrl[i] = Real<T>::nan();
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {   // dataToState of the zero state
        a.obs[k * ld + i] = clampt(path[k] * P.inv_3L, T(-1), T(1));
        a.obs[(3 + k) * ld + i] = clampt(path[3 + k] * P.inv_3L, T(-1), T(1));
        a.obs[(6 + k) * ld + i] = wrap_angle_exact(P.inv_ang, T(0), ang[k]).obs;
    }
}

// ---------------------------------------------------------------------------
// K1: fused env step.  action -> (set-point) -> n_sub x RK4 in registers ->
// wrap -> observation -> done -> reward -> auto-reset.
// V = float / double: one environment per thread.  V = F2: two fp32 environments
// per thread (2t, 2t + 1) on the packed FFMA2 path; loads / stores are 8-byte
// vectors, the (cheap, branchy) epilogue runs per lane.
// ---------------------------------------------------------------------------
// A 64-thread / 128-register "small-shard" shape (16 warps per SM, every warp of a 131 072-environment shard resident at
// once) was measured in round 2 and rejected: 33.4 us per step against 31.0 us with this shape - a warp needs ~18 us for one
// env step whatever the load (8 sub-steps of ~560 dependent-ish packed instructions), so a launch this small is bound by
// that latency and by the synchronised phases of a single wave, not by occupancy (gpurun_out/r2b, DESIGN.md section 8).
template <typename V> struct StepLaunch { static constexpr int BLOCK = 128, MINB = 1; };
// two environments per thread: <= 168 registers, 3 CTAs = 12 warps per SM (measured best, profiles/ r1e notes)
template <> struct StepLaunch<F2> { static constexpr int BLOCK = 128, MINB = 3; };

// SoA element access for one thread: environments i0 .. i0 + L - 1 of row p
template <typename V, typename S> __device__ __forceinline__ V load_v(const S* p, long i0, bool pair) {
    if constexpr (VT<V>::L == 1) { (void)pair; return p[i0]; }
    else { if (pair) return f2_from(*reinterpret_cast<const float2*>(p + i0)); return F2(p[i0], 0.0f); }
}
// asynchronous global -> shared copy of one thread's element(s) of a row (4 / 8 bytes)
template <typename V, typename S> __device__ __forceinline__ void cp_async_v(V* smem, const S* gmem, bool pair) {
    const unsigned dst = (unsigned)__cvta_generic_to_shared(smem);
    if (sizeof(V) == 8 && (VT<V>::L == 1 || pair)) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(gmem));
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(gmem));
}

template <typename V, typename S> __device__ __forceinline__ void store_v(S* p, long i0, bool pair, V x) {
    if constexpr (VT<V>::L == 1) { (void)pair; p[i0] = x; }
    else { if (pair) *reinterpret_cast<float2*>(p + i0) = x.v; else p[i0] = x.v.x; }
}

// CONSTP (fp32, default sparsity): the vehicle constants are the COMPILE-TIME copy of the default BlueROV2 Heavy
// (rov6_default_consts.h) instead of the kernel argument.  The ~130 distinct constants of a set-point stage do not fit the
// 63 uniform registers, so the run-time version reloads them (173 LDCU per sub-step, 8 % of the issue slots, and the
// loop body grows past the 32 KB instruction cache); as literals they become immediates: set-point loop 2044 -> 1818
// instructions, force 1449 -> 1326.  The host selects this instantiation only when the handle's constants equal the
// compiled-in ones bit for bit (mvrl_rov6_create), so the results are identical to the run-time version.
template <typename V, int MODE, bool SP, bool FAST, bool CONSTP = false>
__global__ void __launch_bounds__(StepLaunch<V>::BLOCK, StepLaunch<V>::MINB)
rov6_step_kernel(const __grid_constant__ Rov6StepArgs<typename VT<V>::S> a) {
    using T = typename VT<V>::S;
    constexpr int L = VT<V>::L;
    const long i0 = ((long)blockIdx.x * blockDim.x + threadIdx.x) * L;
    if (i0 >= a.n) return;
    const bool pair = (L == 2) && (i0 + 1 < a.n);   // second lane holds a real environment
    static_assert(!CONSTP || (sizeof(T) == 4 && SP), "compile-time constants exist for the fp32 default vehicle only");
    constexpr Rov6Dev<float> kDefault = MVRL_ROV6_DEFAULT_INIT_F32;
    const auto& P = [&]() -> const Rov6Dev<T>& { if constexpr (CONSTP) return kDefault; else return a.P; }();
    const long ld = a.ld;
    // fp32 without fast-math: pose by compensated summation, trigonometry of stages 2-4 from the stage-1 anchor, and in
    // set-point mode the PID's e - eOld from pose increments (see the RK4 loop and pid6_core_dp)
    constexpr bool ACCURATE_F32 = (sizeof(T) == 4) && !FAST;

    // rows of one array are ld elements apart: walk a byte pointer instead of forming base + k * ld + i0 per row.  The second
    // environment of an unpaired thread (odd batch) reads the row's padding element: rows are padded to an even ld >= n + 1.
    const long row_bytes = ld * (long)sizeof(T);
    auto walk = [&](const T* base, V* dst, int rows) {
        if constexpr (L == 2) {
            const char* p = reinterpret_cast<const char*>(base + i0);
#pragma unroll
            for (int k = 0; k < rows; ++k, p += row_bytes) dst[k] = f2_from(*reinterpret_cast<const float2*>(p));
        } else {   // one environment per thread: indexed rows measured faster (r1_walk)
#pragma unroll
            for (int k = 0; k < rows; ++k) dst[k] = base[k * ld + i0];
        }
    };
    V y[12];
    walk(a.state, y, 12);

    constexpr int NA = (MODE == ACT_RPM) ? 8 : 6;
    V act[NA];
    walk(a.action, act, NA);
    // Needed by the epilogue only: the way-points are copied global -> shared with cp.async (LDGSTS) now, so their
    // DRAM latency hides behind the RK4 loop without holding 6 (12) registers across it - as registers they were
    // spilled (r1i profile: STL in the prologue and LDL / long-scoreboard stalls in the epilogue).
    __shared__ V s_path[6][StepLaunch<V>::BLOCK];
    __shared__ uint32_t s_episode[StepLaunch<V>::BLOCK][L];   // read by the auto-reset only: one environment in max_steps
    if (a.auto_reset) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(&s_episode[threadIdx.x][0]);
        if (L == 2) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(a.episode + i0));
        else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(a.episode + i0));
    }
    {
        const char* p = reinterpret_cast<const char*>(a.path + i0);
#pragma unroll
        for (int k = 0; k < 6; ++k, p += row_bytes) cp_async_v<V>(&s_path[k][threadIdx.x], reinterpret_cast<const T*>(p), (L == 2) || pair);
    }
    int istep_in[L];
#pragma unroll
    for (int l = 0; l < L; ++l) istep_in[l] = 0;
    if constexpr (L == 2) {   // both counters in one 8-byte load (an unpaired thread reads, and ignores, the padding / neighbour)
        const int2 q = *reinterpret_cast<const int2*>(a.istep + i0);
        istep_in[0] = q.x; istep_in[L - 1] = q.y;
    } else {
        istep_in[0] = a.istep[i0];
    }

    V sp[6];
    V e_old[6], e_int[6];
    if constexpr (MODE == ACT_SETPOINT) {
        if (a.fixed_sp) {
#pragma unroll
            for (int k = 0; k < 6; ++k) sp[k] = load_v<V>(a.setpoint + k * ld, i0, pair);
        } else {  // 6DoF.py:545-552
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                sp[k] = fmaf_t(act[k], V(P.act_pos), y[k]);
                sp[3 + k] = fmaf_t(act[3 + k], V(P.act_ang), y[3 + k]);
            }
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) { e_old[k] = load_v<V>(a.ctrl + k * ld, i0, pair); e_int[k] = load_v<V>(a.ctrl + (6 + k) * ld, i0, pair); }
    } else {
#pragma unroll
        for (int k = 3; k < 6; ++k) sp[k] = load_v<V>(a.setpoint + k * ld, i0, pair);
    }

    // fp32 set-point mode: the PID's e - eOld comes from the pose increments between consecutive calls (pid6_core_dp)
    constexpr bool DPOSE = (MODE == ACT_SETPOINT) && ACCURATE_F32;
    V dpose[6], off[6];   // pose of this call - pose of the previous call; offset of this call's pose from y
    if constexpr (MODE == ACT_SETPOINT) {
        const V pose0[6] = {y[0], y[1], y[2], y[3], y[4], y[5]};
        pid6_prime(e_old, sp, pose0);
        if constexpr (DPOSE) {   // first call of the env step: the set-point has moved, the literal e - eOld is the right one
            V e0[6];
            pid6_error(sp, pose0, e0);
#pragma unroll
            for (int k = 0; k < 6; ++k) { dpose[k] = e_old[k] - e0[k]; off[k] = V(T(0)); }
        }
    }

    V H[6];       // thruster wrench of the current evaluation
    V gcf[6];     // generalisedControlForces of the last evaluation
    V dem[8];     // allocated demand (N) of the last evaluation
    if constexpr (MODE == ACT_RPM) {
        V F[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) F[k] = thruster_force(P, act[k]);
        thrust_wrench<V, SP>(P, F, H);  // rpm is held over the env step: hoisted out of RK4
    } else if constexpr (MODE == ACT_FORCE) {
#pragma unroll
        for (int k = 0; k < 6; ++k) gcf[k] = act[k];
    }

    // one derivative evaluation; half = 1 where t - tOld of the PID is h/2, 0 where it is 0 (the only two values inside a step)
    auto f = [&](const Trig6<V>& g, const V (&s)[12], V (&k)[12], int half) {
        const V nu[6] = {s[6], s[7], s[8], s[9], s[10], s[11]};
        if constexpr (MODE != ACT_RPM) {
            if constexpr (MODE == ACT_SETPOINT) {
                const V pose[6] = {s[0], s[1], s[2], s[3], s[4], s[5]};
                if constexpr (DPOSE) {
                    if (half) pid6_core_dp<true>(P, e_old, e_int, sp, pose, dpose, a.pid_kd_inv_dt[1], a.pid_half_dt[1], gcf);
                    else pid6_core_dp<false>(P, e_old, e_int, sp, pose, dpose, a.pid_kd_inv_dt[0], a.pid_half_dt[0], gcf);
                } else pid6_core<false>(P, e_old, e_int, sp, pose, a.pid_inv_dt[half], a.pid_half_dt[half], gcf);
            }
            allocate_demand<V, SP>(P, g, gcf, dem);
            // fp64 used to take the literal route here as well (demand -> sqrt -> rpm -> limit -> thrust law): 8 DSQRT per
            // stage, 22 % of the fp64 set-point kernel's instructions.  F(rpm(c)) = c is an identity up to one rounding, and
            // the limits move to force space exactly (f_max, f_db from the host), so both precisions use it; K2 (derivs)
            // keeps the literal chain because it reports the rpm.
            V F[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) F[j] = demand_to_force(P, dem[j]);
            thrust_wrench<V, SP>(P, F, H);
        }
        V ed[6], acc[6], rhs[6];
        kinematics6<V, FAST>(g, nu, ed);
        body_accel<V, SP>(P, g, nu, H, acc, rhs);
#pragma unroll
        for (int j = 0; j < 6; ++j) { k[j] = ed[j]; k[6 + j] = acc[j]; }
    };

    // classic RK4, y' = y + h/6 (k1 + 2 k2 + 2 k3 + k4).  Velocities (damped, self-correcting) are
    // accumulated as (((y + h/6 k1) + h/3 k2) + h/3 k3) + h/6 k4: one FMA per state and stage.  The
    // pose (pure integrators: every rounding error stays) is advanced in fp32 by the separately
    // summed increment with a Kahan carry across the sub-steps, i.e. about one rounding at ulp(y)
    // per env step instead of 4 n_sub (rk4_pose_update; keeps 1000-step fp32 trajectories within 1e-4).
    // fp32 trigonometry: full sin/cos once per sub-step (stage 1); stages 2-4 sit at angle + c_k k,
    // a small known offset, and use the addition theorem (sincos_delta) unless the offset is large.
    const T h = a.h, hh = a.hh, h6 = a.h6, h3 = a.h3;
    V carry[6];
#pragma unroll
    for (int j = 0; j < 6; ++j) carry[j] = V(T(0));
    for (int sub = 0; sub < a.n_sub; ++sub) {
        V k[12], acc[12], yt[12];
        Trig6<V> g0;
#pragma unroll
        for (int j = 0; j < 12; ++j) { acc[j] = (ACCURATE_F32 && j < 6) ? V(T(0)) : y[j]; yt[j] = y[j]; }
        // the four stages unrolled: measured faster than the rolled loop in every mode (r1r, r2a)
#pragma unroll 4
        for (int st = 0; st < 4; ++st) {
            Trig6<V> g;
            if constexpr (ACCURATE_F32) {
                if (st == 0) {
                    g0 = trig6<V, FAST>(y[3], y[4], y[5]);
                    g = g0;
                } else {
                    const T cp = (st == 3) ? h : hh;          // this stage's state is y + cp * k(previous stage)
                    V d0, d1, d2;
                    if constexpr (DPOSE) { d0 = off[3]; d1 = off[4]; d2 = off[5]; }   // the same products, already formed
                    else { d0 = V(cp) * k[3]; d1 = V(cp) * k[4]; d2 = V(cp) * k[5]; }
                    const V z0 = d0 * d0, z1 = d1 * d1, z2 = d2 * d2;
                    const V zs = z0 + z1 + z2;
                    sincos_delta(g0.sph, g0.cph, d0, z0, &g.sph, &g.cph);
                    sincos_delta(g0.sth, g0.cth, d1, z1, &g.sth, &g.cth);
                    sincos_delta(g0.sps, g0.cps, d2, z2, &g.sps, &g.cps);
                    const auto big = vgt(zs, V(MVRL_TRIG_DELTA_MAX2));   // (NaN offsets stay on the cheap path and stay NaN)
                    if (vany(big)) {   // rare: an environment with a large offset gets the full evaluation - decided per
                                       // environment, so a result never depends on which environment shares the thread
                        const Trig6<V> gf = trig6<V, FAST>(yt[3], yt[4], yt[5]);
                        g.sph = vsel(big, gf.sph, g.sph); g.cph = vsel(big, gf.cph, g.cph);
                        g.sth = vsel(big, gf.sth, g.sth); g.cth = vsel(big, gf.cth, g.cth);
                        g.sps = vsel(big, gf.sps, g.sps); g.cps = vsel(big, gf.cps, g.cps);
                    }
                }
            } else {
                g = trig6<V, FAST>(yt[3], yt[4], yt[5]);
            }
            f(g, yt, k, st & 1);
            const T wk = (st == 0 || st == 3) ? h6 : h3;
            const T ck = (st == 2) ? h : hh;
#pragma unroll
            for (int j = 0; j < 12; ++j) {
                acc[j] = fmaf_t(V(wk), k[j], acc[j]);
                if (DPOSE && j < 6) {
                    // next call's pose is y + o (stages 2-4) or y + the RK4 increment (first stage of the next sub-step)
                    const V o = (st < 3) ? V(ck) * k[j] : acc[j];
                    dpose[j] = (st == 0) ? o : o - off[j];   // the first stage sits at y itself: its offset is 0
                    off[j] = o;
                    if (st < 3) yt[j] = y[j] + o;
                } else if (st < 3) {
                    yt[j] = fmaf_t(V(ck), k[j], y[j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 12; ++j) {
            if (ACCURATE_F32 && j < 6) rk4_pose_update(y[j], carry[j], acc[j]);
            else y[j] = acc[j];
        }
    }

    // ---- epilogue: wrap, observe, done, stats - straight-line for every environment of the thread; the
    // auto-reset of a terminated environment is an out-of-line fix-up AFTER the regular stores (it overwrites
    // that environment's rows; same thread, so program order makes the later stores win) ----
    cp_async_wait_all();     // each thread reads back only its own slots: no barrier needed
    V path_v[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) path_v[k] = s_path[k][threadIdx.x];
    V nonfinite = V(T(0));   // sum of 0 * y_k: 0 when every state is finite, NaN otherwise
#pragma unroll
    for (int k = 0; k < 12; ++k) nonfinite = fmaf_t(y[k], V(T(0)), nonfinite);
    V obs_v[9];
    V pos_v[6];   // (way-point - position) / (3 Length), 6DoF.py:470-476, for every environment of the thread at once
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        pos_v[k] = (path_v[k] - y[k]) * V(P.inv_3L);
        pos_v[3 + k] = (path_v[3 + k] - y[k]) * V(P.inv_3L);
    }
    int n_done_t = 0, len_t = 0, n_bad_t = 0;
    bool reset_lane[L], lane_on[L], ok[L];
    int istep[L];
    unsigned char done_flag[L];
    T ang_raw[L][3], spa[L][3];
    // phase A - wrap (6DoF.py:560) and dataToState (467-483) on the fast path, for every environment of the thread at once
    // on the value type (packed for two environments): a wrapped angle is the angle plus a whole number of turns chosen by
    // two 0 / 1 masks, an angle error the difference plus the turns that bring it into [-pi, pi) (see angle_error_v), and
    // all clamps are min / max pairs.  Valid while every angle is inside (-2 pi, 4 pi) and every difference inside
    // (-2 pi, 2 pi): ONE test per environment at the end; phase B redoes the rest with the exact out-of-line functions.
    const V tp = V(T(MVRL_TWO_PI));
    V ang_lo = y[3], ang_hi = y[3], d_worst = V(T(0)), ang_big = V(T(0));
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const V ang = y[3 + k];
#pragma unroll
        for (int l = 0; l < L; ++l) { ang_raw[l][k] = lane_get(ang, l); spa[l][k] = lane_get(sp[3 + k], l); }
        ang_lo = tmin(ang_lo, ang); ang_hi = tmax(ang_hi, ang); ang_big = tmax(ang_big, tabs(ang));
        const V wrapped = fmaf_t(tp, vmask_lt(ang, V(T(0))) - vmask_ge(ang, tp), ang);
        const V d = sp[3 + k] - wrapped;
        d_worst = tmax(d_worst, tabs(d));
        const V ae = fmaf_t(tp, vmask_lt(d, V(T(-MVRL_PI))) - vmask_ge(d, V(T(MVRL_PI))), d);
        y[3 + k] = wrapped;
        obs_v[k] = tmax(V(T(-1)), tmin(V(T(1)), pos_v[k]));
        obs_v[3 + k] = tmax(V(T(-1)), tmin(V(T(1)), pos_v[3 + k]));
        obs_v[6 + k] = tmax(V(T(-1)), tmin(V(T(1)), ae * V(P.inv_ang)));
    }
#pragma unroll
    for (int l = 0; l < L; ++l) {
        lane_on[l] = (l == 0) || pair;
        istep[l] = istep_in[l] + 1;
        bool bad = lane_get(nonfinite, l) != T(0);   // NaN compares unequal
        if constexpr (sizeof(T) == 4 && !FAST) {  // outside the exact range of the fp32 sin/cos reduction
            bad = bad || lane_get(ang_big, l) > T(MVRL_SINCOS_F32_MAX_ARG);
        }
        // all three comparisons are false for NaN: the exact path then propagates it
        ok[l] = (lane_get(ang_lo, l) > T(-MVRL_TWO_PI) && lane_get(ang_hi, l) < T(2 * MVRL_TWO_PI) && lane_get(d_worst, l) < T(MVRL_TWO_PI)) || !lane_on[l];
        const bool is_done = istep[l] >= a.max_steps;  // 6DoF.py:569-571
        reset_lane[l] = lane_on[l] && is_done && a.auto_reset;
        n_done_t += reset_lane[l] ? 1 : 0;
        len_t += reset_lane[l] ? istep[l] : 0;
        n_bad_t += (lane_on[l] && bad) ? 1 : 0;
        done_flag[l] = is_done ? 1 : 0;
        if constexpr (MODE == ACT_SETPOINT) { if (lane_on[l]) a.ctrl[12 * ld + i0 + l] = T(istep[l]) * a.dt; }
    }
    if constexpr (L == 2) {   // done flags and counters of a paired thread go out as one 2-byte and one 8-byte store
        if (pair) {
            *reinterpret_cast<uchar2*>(a.done + i0) = make_uchar2(done_flag[0], done_flag[L - 1]);
            *reinterpret_cast<int2*>(a.istep + i0) = make_int2(istep[0], istep[L - 1]);
        } else {
            a.done[i0] = done_flag[0];
            a.istep[i0] = istep[0];
        }
    } else {
        a.done[i0] = done_flag[0];
        a.istep[i0] = istep[0];
    }
    // phase B - rare: an angle outside the fast range goes through the exact, out-of-line modulo
    bool all_ok = true;
#pragma unroll
    for (int l = 0; l < L; ++l) all_ok = all_ok && ok[l];
    if (!all_ok) {
#pragma unroll
        for (int l = 0; l < L; ++l) {
            if (ok[l]) continue;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const WrapObs<T> r = wrap_angle_exact(P.inv_ang, ang_raw[l][k], spa[l][k]);
                lane_set(y[3 + k], l, r.wrapped);
                lane_set(obs_v[6 + k], l, r.obs);
            }
        }
    }
    if (a.aux != nullptr) {  // what the reference logs per step, 6DoF.py:578-580
#pragma unroll
        for (int l = 0; l < L; ++l) {
            if (!lane_on[l]) continue;
            const long i = i0 + l;
            if constexpr (MODE == ACT_RPM) {
#pragma unroll
                for (int k = 0; k < 6; ++k) a.aux[k * ld + i] = T(0);
#pragma unroll
                for (int k = 0; k < 8; ++k) a.aux[(6 + k) * ld + i] = lane_get(act[k], l);
            } else {
#pragma unroll
                for (int k = 0; k < 6; ++k) a.aux[k * ld + i] = lane_get(gcf[k], l);
#pragma unroll
                for (int k = 0; k < 8; ++k) a.aux[(6 + k) * ld + i] = demand_to_rpm(P, T(lane_get(dem[k], l)));
            }
        }
    }

    if (a.stats != nullptr) stats_accumulate_counts(a.stats, n_done_t, len_t, n_bad_t);
    auto walk_out = [&](T* base, const V* src, int rows) {   // same pointer walk for the stores; the unpaired thread stores one element
        if constexpr (L == 2) {
            char* p = reinterpret_cast<char*>(base + i0);
#pragma unroll
            for (int k = 0; k < rows; ++k, p += row_bytes) {
                if (pair) *reinterpret_cast<float2*>(p) = src[k].v; else *reinterpret_cast<float*>(p) = src[k].v.x;
            }
        } else {
#pragma unroll
            for (int k = 0; k < rows; ++k) base[k * ld + i0] = src[k];
        }
    };
    walk_out(a.state, y, 12);
    walk_out(a.obs, obs_v, 9);
    store_v<V>(a.reward, i0, pair, V(T(0)));  // 6DoF.py:575
    if constexpr (MODE == ACT_SETPOINT) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            store_v<V>(a.setpoint + k * ld, i0, pair, sp[k]);
            store_v<V>(a.ctrl + k * ld, i0, pair, e_old[k]);
            store_v<V>(a.ctrl + (6 + k) * ld, i0, pair, e_int[k]);
        }
    }
#pragma unroll
    for (int l = 0; l < L; ++l) {
        if (reset_lane[l]) rov6_auto_reset_env<T, MODE>(a, i0 + l, s_episode[threadIdx.x][l]);
    }
}

// ---------------------------------------------------------------------------
// K2: one derivative evaluation per environment, with optional dump of RHS,
// controller forces, rpm and the retComp columns.
// ---------------------------------------------------------------------------
template <typename T> struct Rov6DerivArgs {
    Rov6Dev<T> P;
    long n, ld;
    const T* state; const T* act; const T* t; const T* setpoint; T* ctrl; T* dstate; T* aux;
};

template <typename T, int MODE, bool SP>
__global__ void __launch_bounds__(128)
rov6_derivs_kernel(const __grid_constant__ Rov6DerivArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const Rov6Dev<T>& P = a.P;
    const long ld = a.ld;
    T s[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) s[k] = a.state[k * ld + i];
    const Trig6<T> g = trig6<T, false>(s[3], s[4], s[5]);
    const T nu[6] = {s[6], s[7], s[8], s[9], s[10], s[11]};
    T gcf[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
    T rpm[8];
    T F[8], H[6];
    if constexpr (MODE == ACT_RPM) {
#pragma unroll
        for (int k = 0; k < 8; ++k) { rpm[k] = a.act[k * ld + i]; F[k] = thruster_force(P, rpm[k]); }
    } else {
        if constexpr (MODE == ACT_FORCE) {
#pragma unroll
            for (int k = 0; k < 6; ++k) gcf[k] = a.act[k * ld + i];
        } else {
            T e_old[6], e_int[6], sp[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                e_old[k] = a.ctrl[k * ld + i]; e_int[k] = a.ctrl[(6 + k) * ld + i]; sp[k] = a.setpoint[k * ld + i];
            }
            const T t = a.t[i];
            const T dtc = t - a.ctrl[12 * ld + i];
            const T pose[6] = {s[0], s[1], s[2], s[3], s[4], s[5]};
            pid6(P, e_old, e_int, sp, pose, dtc, gcf);
#pragma unroll
            for (int k = 0; k < 6; ++k) { a.ctrl[k * ld + i] = e_old[k]; a.ctrl[(6 + k) * ld + i] = e_int[k]; }
            a.ctrl[12 * ld + i] = t;
        }
        T dem[8];
        allocate_demand<T, SP>(P, g, gcf, dem);
#pragma unroll
        for (int k = 0; k < 8; ++k) { rpm[k] = demand_to_rpm(P, dem[k]); F[k] = thruster_force(P, rpm[k]); }
    }
    thrust_wrench<T, SP>(P, F, H);
    T ed[6], acc[6], rhs[6];
    kinematics6<T, false>(g, nu, ed);
    body_accel<T, SP>(P, g, nu, H, acc, rhs, a.aux ? a.aux + 20 * ld + i : nullptr, ld);
#pragma unroll
    for (int k = 0; k < 6; ++k) { a.dstate[k * ld + i] = ed[k]; a.dstate[(6 + k) * ld + i] = acc[k]; }
    if (a.aux != nullptr) {
#pragma unroll
        for (int k = 0; k < 6; ++k) { a.aux[k * ld + i] = rhs[k]; a.aux[(6 + k) * ld + i] = gcf[k]; }
#pragma unroll
        for (int k = 0; k < 8; ++k) a.aux[(12 + k) * ld + i] = rpm[k];
    }
}

// ---------------------------------------------------------------------------
// reset (6DoF.py:485-529)
// ---------------------------------------------------------------------------
template <typename T> struct Rov6ResetArgs {
    Rov6Dev<T> P;
    long n, ld;
    T* state; T* obs; int32_t* istep; T* setpoint; T* path; T* ctrl; const uint32_t* episode; T* aux;
    const uint8_t* mask;
    T init_sp[6];
    int has_init_sp;
    unsigned long long seed, env_id0;
};

template <typename T>
__global__ void __launch_bounds__(128)
rov6_reset_kernel(const __grid_constant__ Rov6ResetArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if (a.mask != nullptr && a.mask[i] == 0) return;
    const long ld = a.ld;
    T y[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) { y[k] = T(0); a.state[k * ld + i] = T(0); }  // 6DoF.py:517-519
    a.istep[i] = 0;
    T path[6], sp[6];
    if (a.has_init_sp) {  // 6DoF.py:502-511
#pragma unroll
        for (int k = 0; k < 6; ++k) sp[k] = a.init_sp[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) { path[k] = sp[k]; path[3 + k] = sp[k]; }
    } else {
        const uint32_t ep = a.episode ? a.episode[i] : 0u;
        const Reset6<T> rs = draw_reset6<T>(a.seed, a.env_id0 + (unsigned long long)i, ep);
#pragma unroll
        for (int k = 0; k < 6; ++k) path[k] = rs.path[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) { sp[k] = path[k]; sp[3 + k] = rs.orient[k]; }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k) { a.path[k * ld + i] = path[k]; a.setpoint[k * ld + i] = sp[k]; }
    if (a.ctrl != nullptr) {
#pragma unroll
        for (int k = 0; k < 13; ++k) a.ctrl[k * ld + i] = T(0);
        a.ctrl[i] = Real<T>::nan();
    }
    if (a.aux != nullptr) {
#pragma unroll
        for (int k = 0; k < 14; ++k) a.aux[k * ld + i] = T(0);
    }
    const T spa[3] = {sp[3], sp[4], sp[5]};
    T obs[9];
    observe6(a.P, y, path, spa, obs);
#pragma unroll
    for (int k = 0; k < 9; ++k) a.obs[k * ld + i] = obs[k];
}

// ---------------------------------------------------------------------------
// stand-alone PID (6DoF.py:43-73)
// ---------------------------------------------------------------------------
template <typename T> struct Rov6PidArgs {
    Rov6Dev<T> P;
    long n, ld;
    const T* pose; const T* t; const T* setpoint; T* ctrl; T* forces;
};

template <typename T>
__global__ void __launch_bounds__(128)
rov6_pid_kernel(const __grid_constant__ Rov6PidArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const long ld = a.ld;
    T e_old[6], e_int[6], sp[6], pose[6], out[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        e_old[k] = a.ctrl[k * ld + i]; e_int[k] = a.ctrl[(6 + k) * ld + i];
        sp[k] = a.setpoint[k * ld + i]; pose[k] = a.pose[k * ld + i];
    }
    const T t = a.t[i];
    pid6(a.P, e_old, e_int, sp, pose, t - a.ctrl[12 * ld + i], out);
#pragma unroll
    for (int k = 0; k < 6; ++k) { a.ctrl[k * ld + i] = e_old[k]; a.ctrl[(6 + k) * ld + i] = e_int[k]; a.forces[k * ld + i] = out[k]; }
    a.ctrl[12 * ld + i] = t;
}

}  // namespace mvrl
