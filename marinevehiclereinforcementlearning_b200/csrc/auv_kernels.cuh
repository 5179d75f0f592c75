// Legacy "verySimpleAuv" env step (K4) and turbulence-field interpolation.
// Restates tag_00_Dec2023_simpleControlTurbulence/verySimpleAuv.py:147-410 and
// flowGenerator.py:53-136.  One environment per thread.
#pragma once
#include "mvrl_math.cuh"
#include "rov6_kernels.cuh"  // stats_accumulate

namespace mvrl {

// Scaled flow field on the device: [nt][ny][nx][NC] (NC = 3: u, v, Cp as in the
// reference; NC = 2: u, v only, the copy the env kernel gathers from).
template <typename T> struct FlowDev {
    const T* field;
    int nt, ny, nx, nc;
    T dx, dy, dt;
    T inv_dx, inv_dy, inv_dt;   // host-computed reciprocals (step kernel: three multiplies instead of three IEEE divisions)
};

// flowGenerator.py:97-136: trilinear interpolation, indices clamped to the grid,
// weights NOT clamped (extrapolation outside, and `translate` is ignored).
template <typename T> struct FlowCell { int kk, jj, ii; T wt, wx, wy; };

// RCP = true (env step kernel): grid coordinates by multiplication with the host's reciprocals.  The result differs from
// the quotient by at most one rounding; the interpolant is continuous across cell faces, so even a coordinate that lands on
// the other side of a face changes the value by ~1 ulp.  The stand-alone interp entry keeps the reference's divisions.
template <bool RCP = false, typename T>
__device__ __forceinline__ FlowCell<T> flow_locate(const FlowDev<T>& f, T time, T x, T y) {
    const T tt = RCP ? time * f.inv_dt : time / f.dt, xx = RCP ? x * f.inv_dx : x / f.dx, yy = RCP ? y * f.inv_dy : y / f.dy;
    FlowCell<T> c;
    // clamp in floating point first: int conversion of huge / non-finite values is undefined.  fmin / fmax
    // return the non-NaN operand, so a NaN coordinate (a vehicle that diverged) indexes cell 0 and yields NaN
    // weights instead of an out-of-bounds gather (upstream raises on int(floor(nan))).
    c.kk = (int)fmin(T(f.nt - 2), fmax(T(0), Real<T>::floor(tt)));
    c.ii = (int)fmin(T(f.nx - 2), fmax(T(0), Real<T>::floor(xx)));
    c.jj = (int)fmin(T(f.ny - 2), fmax(T(0), Real<T>::floor(yy)));
    c.wt = tt - T(c.kk); c.wx = xx - T(c.ii); c.wy = yy - T(c.jj);
    return c;
}

// weights applied in the reference's order: along x, then y, then time
template <typename T>
__device__ __forceinline__ T flow_blend(const FlowCell<T>& c, T c000, T c001, T c010, T c011, T c100, T c101, T c110, T c111) {
    const T r00 = c000 * (T(1) - c.wx) + c001 * c.wx, r01 = c010 * (T(1) - c.wx) + c011 * c.wx;
    const T r10 = c100 * (T(1) - c.wx) + c101 * c.wx, r11 = c110 * (T(1) - c.wx) + c111 * c.wx;
    return ((T(1) - c.wy) * r00 + c.wy * r01) * (T(1) - c.wt) + ((T(1) - c.wy) * r10 + c.wy * r11) * c.wt;
}

// Gathers 8 corners x NOUT components straight from L2 (read-only path).
template <typename T, int NOUT>
__device__ __forceinline__ void flow_interp(const FlowDev<T>& f, T time, T x, T y, T (&res)[NOUT]) {
    const FlowCell<T> c = flow_locate(f, time, x, y);
    const long row = (long)f.nx * f.nc, plane = (long)f.ny * row;
    const T* p = f.field + (long)c.kk * plane + (long)c.jj * row + (long)c.ii * f.nc;
#pragma unroll
    for (int k = 0; k < NOUT; ++k) {
        const T* q = p + k;
        res[k] = flow_blend(c, __ldg(q), __ldg(q + f.nc), __ldg(q + row), __ldg(q + row + f.nc),
                            __ldg(q + plane), __ldg(q + plane + f.nc), __ldg(q + plane + row), __ldg(q + plane + row + f.nc));
    }
}

// The env's gather, nc = 2 (u, v interleaved): every corner is one 8-byte element and the two x-neighbours
// are adjacent, so a cell is 4 rows of 16 contiguous bytes.  Each thread stages its rows into its own shared
// memory slot with cp.async (LDGSTS: no register round trip, the copies stay in flight while the thread
// works through the 30-float action ring), then blends from shared memory.
constexpr int AUV_BLOCK = 128;   // measured: 64 threads per block +1 % (noise level), 256 threads -18 % (r1_auvblk)

__device__ __forceinline__ void cp_async8(void* smem, const void* gmem) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}

// issue: 8 x 8-byte copies (2 time levels x 2 rows x 2 x-neighbours) into slot[8] of this thread
__device__ __forceinline__ void flow_stage_issue(const FlowDev<float>& f, const FlowCell<float>& c, float2 (*slot)[AUV_BLOCK]) {
    const long row = (long)f.nx, plane = (long)f.ny * row;   // in float2 elements
    const float2* p = reinterpret_cast<const float2*>(f.field) + (long)c.kk * plane + (long)c.jj * row + c.ii;
#pragma unroll
    for (int dk = 0; dk < 2; ++dk)
#pragma unroll
        for (int dj = 0; dj < 2; ++dj)
#pragma unroll
            for (int di = 0; di < 2; ++di) cp_async8(&slot[dk * 4 + dj * 2 + di][threadIdx.x], p + dk * plane + dj * row + di);
}

__device__ __forceinline__ void flow_stage_blend(const FlowCell<float>& c, float2 (*slot)[AUV_BLOCK], float (&res)[2]) {
    float2 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = slot[k][threadIdx.x];
    res[0] = flow_blend(c, v[0].x, v[1].x, v[2].x, v[3].x, v[4].x, v[5].x, v[6].x, v[7].x);
    res[1] = flow_blend(c, v[0].y, v[1].y, v[2].y, v[3].y, v[4].y, v[5].y, v[6].y, v[7].y);
}

template <typename T> struct AuvDev {
    T m, Izz, Xuu, Yvv, Nrr, Xu, Yv, Nr, maxForce, maxMoment;
    T xmin, xmax, ymin, ymax;
    T noise_coeffs, noise_act;
    T t_quarter;  // flow.time[nt // 4], upper bound of the random flow time offset
    // AuvEnvCyl (verySimpleAuv_cyl.py:29-41): way-points x, y, target heading; switch radius
    int cyl, n_wp;
    T wp_thr;
    T wp[32][3];
};

template <typename T> struct AuvStepArgs {
    AuvDev<T> P;
    FlowDev<T> flow;
    long n, ld;
    T* state;        // [6][ld] x y psi u v r
    const T* action; // [3][ld]
    T* obs;          // [11][ld]
    T* reward; uint8_t* done; int32_t* istep;
    T* mults;        // [11][ld] m I Xuu Yvv Nrr Xu Yv Nr Xact Yact Nact
    T* target;       // [2][ld] headingTarget, flowDataTimeOffset
    T* err_o;        // [3][ld] perr_o x, perr_o y, herr_o
    T* recent;       // [30][ld] ring of the 10 most recent actions (slot = (iStep - 1) % 10)
    T* ep_return;    // [ld] running episode return
    int32_t* iwp;    // [ld] way-point index (AuvEnvCyl only)
    uint32_t* episode; T* term_obs; T* aux; double* stats;
    T dt;
    int max_steps;
    unsigned long long seed, env_id0;
    int auto_reset, stop_on_bounds, apply_noise;
};

// dataToState: V3 of AuvEnv (verySimpleAuv.py:147-214; target at the origin, no scaling) or, for AuvEnvCyl,
// V0 scaling against the current way-point (verySimpleAuv_cyl.py:84-115).  The scales are literals, so they are applied
// as multiplications by their (double-rounded) reciprocals; CYL is a template parameter: the plain env has no scaling
// at all.
template <bool CYL, typename T>
__device__ __forceinline__ void observe_auv(T tx, T ty, T x, T y, T psi, T u, T v, T r, T heading_target, T perr_ox, T perr_oy,
                                            T herr_o, T (&obs)[11]) {
    const T px = tx - x, py = ty - y;
    const T herr = angle_error(heading_target, psi);
    constexpr double pi = 3.14159265358979323846;
    const T isp = CYL ? T(1. / 0.2) : T(1), isdh = CYL ? T(1. / (2. / 180 * pi)) : T(1), isdp = CYL ? T(1. / 0.025) : T(1);
    const T isv = CYL ? T(1. / 0.2) : T(1), isr = CYL ? T(1. / (30. / 180. * pi)) : T(1);
    obs[0] = clampt(CYL ? px * isp : px, T(-1), T(1));
    obs[1] = clampt(CYL ? py * isp : py, T(-1), T(1));
    obs[2] = clampt(herr * T(1. / (45. / 180. * pi)), T(-1), T(1));
    obs[3] = clampt(CYL ? (herr - herr_o) * isdh : herr - herr_o, T(-1), T(1));
    obs[4] = clampt(CYL ? (px - perr_ox) * isdp : px - perr_ox, T(-1), T(1));
    obs[5] = clampt(CYL ? (py - perr_oy) * isdp : py - perr_oy, T(-1), T(1));
    obs[6] = clampt(CYL ? u * isv : u, T(-1), T(1));
    obs[7] = clampt(CYL ? v * isv : v, T(-1), T(1));
    obs[8] = clampt(CYL ? r * isr : r, T(-1), T(1));
    obs[9] = T(0);
    obs[10] = T(0);
}

// reset draws in the reference's order (verySimpleAuv.py:222-245), Philox instead of np.random
template <typename T>
__device__ __forceinline__ void draw_reset_auv(const AuvDev<T>& P, unsigned long long seed, unsigned long long env, uint32_t episode,
                                               bool apply_noise, T (&mults)[11], T* x, T* y, T* heading, T* target, T* offset) {
    uint32_t w[16];
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const uint4 q = Philox::draw(seed, env, episode, 0u, (uint32_t)b);
        w[4 * b] = q.x; w[4 * b + 1] = q.y; w[4 * b + 2] = q.z; w[4 * b + 3] = q.w;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) mults[k] = apply_noise ? T(1) + P.noise_coeffs / T(2) - u01<T>(w[k]) * P.noise_coeffs : T(1);
#pragma unroll
    for (int k = 8; k < 11; ++k) mults[k] = apply_noise ? T(1) + P.noise_act / T(2) - u01<T>(w[k]) * P.noise_act : T(1);
    *x = (u01<T>(w[11]) - T(0.5)) * T(0.5) * (P.xmax - P.xmin);
    *y = (u01<T>(w[12]) - T(0.5)) * T(0.5) * (P.ymax - P.ymin);
    *heading = u01<T>(w[13]) * T(MVRL_TWO_PI);
    if (P.cyl) {   // verySimpleAuv_cyl.py:155-160: the heading target comes from the way-point, one draw fewer
        *offset = u01<T>(w[14]) * P.t_quarter;
    } else {
        *target = u01<T>(w[14]) * T(MVRL_TWO_PI);
        *offset = u01<T>(w[15]) * P.t_quarter;
    }
}

// Everything one environment reads, as values
template <typename T> struct AuvIn {
    T x, y, psi, u, v, r, a0, a1, a2, heading_target, t_offset, err_o0, err_o1, err_o2, ep_return;
    T mm[11];
    T ring[10][3];
    int istep, iwp;
    uint32_t episode;
};

// the two ways the env kernel fetches its 8 flow-field corners: staged through shared memory with cp.async (fp32, 2
// components) or straight from L2
template <typename T> struct GatherDirect {
    const FlowDev<T>& f;
    __device__ __forceinline__ void issue(const FlowCell<T>&) {}
    __device__ __forceinline__ void finish(const FlowCell<T>& c, T (&cur)[2]) {
        const long row = (long)f.nx * f.nc, plane = (long)f.ny * row;
        const T* p = f.field + (long)c.kk * plane + (long)c.jj * row + (long)c.ii * f.nc;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const T* q = p + k;
            cur[k] = flow_blend(c, __ldg(q), __ldg(q + f.nc), __ldg(q + row), __ldg(q + row + f.nc),
                                __ldg(q + plane), __ldg(q + plane + f.nc), __ldg(q + plane + row), __ldg(q + plane + row + f.nc));
        }
    }
};
struct GatherStaged {
    const FlowDev<float>& f;
    float2 (*slot)[AUV_BLOCK];
    __device__ __forceinline__ void issue(const FlowCell<float>& c) {
        flow_stage_issue(f, c, slot);
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
    __device__ __forceinline__ void finish(const FlowCell<float>& c, float (&cur)[2]) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");   // each thread reads back only what it copied itself: no barrier
        flow_stage_blend(c, slot, cur);
    }
};

// K4: AuvEnv.step, verySimpleAuv.py:264-410 - the arithmetic and the stores of ONE environment
template <typename T, bool CYL, typename Gather>
__device__ __forceinline__ void auv_step_env(const AuvStepArgs<T>& a, long i, const AuvIn<T>& in, Gather gather) {
    const AuvDev<T>& P = a.P;
    const long ld = a.ld;
    const long row_bytes = ld * (long)sizeof(T);
    T x = in.x, y = in.y, psi = in.psi, u = in.u, v = in.v, r = in.r;
    const T a0 = in.a0, a1 = in.a1, a2 = in.a2;
    T heading_target = in.heading_target, t_offset = in.t_offset;
    int iwp = 0;
    T tx = T(0), ty = T(0);   // positionTarget: the origin, or the current way-point of AuvEnvCyl
    if constexpr (CYL) { iwp = in.iwp; tx = P.wp[iwp][0]; ty = P.wp[iwp][1]; heading_target = P.wp[iwp][2]; }
    const int istep = in.istep + 1;
    T mm[11];
#pragma unroll
    for (int k = 0; k < 11; ++k) mm[k] = in.mm[k];
    T ring[10][3];
#pragma unroll
    for (int s = 0; s < 10; ++s) {
#pragma unroll
        for (int c = 0; c < 3; ++c) ring[s][c] = in.ring[s][c];
    }
    const T time = T(istep) * a.dt;
    const FlowCell<T> cell = flow_locate<true>(a.flow, time + t_offset, x, y);
    gather.issue(cell);      // the gather (L2) lands while the ring statistics below are set up
    bool is_done = istep >= a.max_steps;

    // recentActions.appendleft(action): ring slot, then statistics over the valid entries
    const int slot = (istep - 1) % 10;
    const int cnt = istep < 10 ? istep : 10;
#pragma unroll
    for (int s = 0; s < 10; ++s) {
        if (s == slot) { ring[s][0] = a0; ring[s][1] = a1; ring[s][2] = a2; }
    }
    a.recent[(slot * 3 + 0) * ld + i] = a0;
    a.recent[(slot * 3 + 1) * ld + i] = a1;
    a.recent[(slot * 3 + 2) * ld + i] = a2;

    const T Fx_set = a0 * P.maxForce * mm[8], Fy_set = a1 * P.maxForce * mm[9], N_set = a2 * P.maxMoment * mm[10];
    T sn, cs;
    Real<T>::sincos(psi, &sn, &cs);
    T cur[2];
    gather.finish(cell, cur);
    const T dxv = u - cur[0], dyv = v - cur[1];
    const T vr0 = cs * dxv + sn * dyv, vr1 = -sn * dxv + cs * dyv;
    const T fh0 = (P.Xu * mm[5] + P.Xuu * mm[2] * tabs(vr0)) * vr0;
    const T fh1 = (P.Yv * mm[6] + P.Yvv * mm[3] * tabs(vr1)) * vr1;
    const T fh2 = (P.Nr * mm[7] + P.Nrr * mm[4] * tabs(r)) * r;
    const T Fx = cs * fh0 - sn * fh1, Fy = sn * fh0 + cs * fh1;
    // one reciprocal per inertia instead of three divisions (<= 1 ulp from the quotients)
    const T inv_m = T(1) / (P.m * mm[0]), inv_i = T(1) / (P.Izz * mm[1]);
    const T ax = (Fx + Fx_set) * inv_m, ay = (Fy + Fy_set) * inv_m, ar = (fh2 + N_set) * inv_i;
    // explicit Euler, position advanced with the OLD velocity (verySimpleAuv.py:321-326)
    x = x + u * a.dt;
    y = y + v * a.dt;
    psi = pymod_pos(psi + r * a.dt, T(MVRL_TWO_PI));
    u = u + ax * a.dt;
    v = v + ay * a.dt;
    r = r + ar * a.dt;

    T obs[11];
    observe_auv<CYL>(tx, ty, x, y, psi, u, v, r, heading_target, in.err_o0, in.err_o1, in.err_o2, obs);

    T bonus = T(0);
    if (x < P.xmin || x > P.xmax) { if (a.stop_on_bounds) is_done = true; bonus += T(-100); }
    if (y < P.ymin || y > P.ymax) { if (a.stop_on_bounds) is_done = true; bonus += T(-100); }
    T perr_x = tx - x, perr_y = ty - y;
    T herr = angle_error(heading_target, psi);
    const T perr_norm = Real<T>::sqrt(perr_x * perr_x + perr_y * perr_y);
    if constexpr (CYL) {
        if (perr_norm < P.wp_thr) {                              // way-point reached (verySimpleAuv_cyl.py:249-253);
            iwp = iwp + 1 < P.n_wp ? iwp + 1 : P.n_wp - 1;      // the errors above stay relative to the OLD target
            tx = P.wp[iwp][0]; ty = P.wp[iwp][1]; heading_target = P.wp[iwp][2];
        }
    }

    // rmsAc: mean over components of the population std of the <= 10 recent actions (:353-355)
    T rms = T(0);
    const T inv_cnt = T(1) / T(cnt);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        T mean = T(0);
#pragma unroll
        for (int s = 0; s < 10; ++s) mean += (s < cnt) ? ring[s][c] : T(0);
        mean *= inv_cnt;
        T var = T(0);
#pragma unroll
        for (int s = 0; s < 10; ++s) { const T d = ring[s][c] - mean; var += (s < cnt) ? d * d : T(0); }
        rms += Real<T>::sqrt(var * inv_cnt);
    }
    rms *= T(1. / 3.);
    const T pi = T(3.14159265358979323846);
    const T herr_deg = tabs(herr * T(180. / 3.14159265358979323846));
    const T t0 = Real<T>::exp(T(-5) * perr_norm);
    // the two branches of verySimpleAuv.py:343-346 are one exponential of a selected argument with a selected sign
    const bool facing = tabs(herr) < pi * T(0.5);
    const T t1e = Real<T>::exp(T(-0.1) * (facing ? herr_deg : T(180) - herr_deg));
    const T t1 = facing ? t1e : -t1e;
    const T t2 = Real<T>::exp(T(-0.6) * rms);
    const T t3 = T(-0.1 / 3.) * (a0 * a0 + a1 * a1 + a2 * a2);
    const T rew = t0 + t1 + t2 + t3 + bonus;
    const T ep_ret = in.ep_return + rew;

    if (a.aux != nullptr) {  // the per-step log columns of verySimpleAuv.py:389-401 that are not state/obs
        const T vals[14] = {Fx, Fy, fh2, Fx_set, Fy_set, N_set, cur[0], cur[1], rms, t0, t1, t2, t3, bonus};
#pragma unroll
        for (int k = 0; k < 14; ++k) a.aux[k * ld + i] = vals[k];
    }
    const bool bad = !(finite_t(x) && finite_t(y) && finite_t(psi) && finite_t(u) && finite_t(v) && finite_t(r));
    if (a.stats != nullptr) stats_accumulate(a.stats, is_done && a.auto_reset, (double)istep, (double)ep_ret, bad);

    int istep_out = istep;
    T ep_ret_out = ep_ret;
    if (is_done && a.auto_reset) {
        if (a.term_obs != nullptr) {
#pragma unroll
            for (int k = 0; k < 11; ++k) a.term_obs[k * ld + i] = obs[k];
        }
        const uint32_t ep = in.episode + 1u;
        a.episode[i] = ep;
        draw_reset_auv(P, a.seed, a.env_id0 + (unsigned long long)i, ep, a.apply_noise != 0, mm, &x, &y, &psi, &heading_target, &t_offset);
#pragma unroll
        for (int k = 0; k < 11; ++k) a.mults[k * ld + i] = mm[k];
        a.target[ld + i] = t_offset;
        u = v = r = T(0);
        istep_out = 0;
        ep_ret_out = T(0);
        perr_x = tx - x; perr_y = ty - y;     // (the way-point index is NOT reset: upstream sets it in __init__ only)
        herr = angle_error(heading_target, psi);
        observe_auv<CYL>(tx, ty, x, y, psi, u, v, r, heading_target, perr_x, perr_y, herr, obs);
    }
    a.target[i] = heading_target;
    if constexpr (CYL) a.iwp[i] = iwp;
    a.state[i] = x; a.state[ld + i] = y; a.state[2 * ld + i] = psi;
    a.state[3 * ld + i] = u; a.state[4 * ld + i] = v; a.state[5 * ld + i] = r;
    a.err_o[i] = perr_x; a.err_o[ld + i] = perr_y; a.err_o[2 * ld + i] = herr;
    {
        char* p = reinterpret_cast<char*>(a.obs + i);
#pragma unroll
        for (int k = 0; k < 11; ++k, p += row_bytes) *reinterpret_cast<T*>(p) = obs[k];
    }
    a.reward[i] = rew;
    a.done[i] = is_done ? 1 : 0;
    a.istep[i] = istep_out;
    a.ep_return[i] = ep_ret_out;
}

// Plain kernel: one environment per thread, every input requested before anything waits on one of them and before the first
// store (the flow-cell lookup stalls on x / y / istep, and whatever is issued after it pays a second DRAM round trip; the
// compiler cannot move a load above a store through pointers it must assume to alias - profiles/ r1t).
// STAGE: the fp32 / 2-component gather goes through shared memory with cp.async (see flow_stage_issue).
// fp32: 5 CTAs of 128 threads per SM (<= 102 registers); fp64 keeps what the compiler needs
template <typename T, bool STAGE, bool CYL>
__global__ void __launch_bounds__(AUV_BLOCK, (sizeof(T) == 4 ? 5 : 1))
auv_step_kernel(const __grid_constant__ AuvStepArgs<T> a) {
    __shared__ float2 stage[STAGE ? 8 : 1][AUV_BLOCK];
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    const long ld = a.ld;
    // rows of one array are ld elements apart: walk a pointer down them instead of forming base + k * ld + i (64-bit
    // multiply-add) for each of the ~125 accesses of this kernel
    const long row_bytes = ld * (long)sizeof(T);
    AuvIn<T> in;
    in.x = a.state[i]; in.y = a.state[ld + i]; in.psi = a.state[2 * ld + i];
    in.heading_target = a.target[i]; in.t_offset = a.target[ld + i];
    in.iwp = CYL ? a.iwp[i] : 0;
    in.istep = a.istep[i];
    in.u = a.state[3 * ld + i]; in.v = a.state[4 * ld + i]; in.r = a.state[5 * ld + i];
    in.a0 = a.action[i]; in.a1 = a.action[ld + i]; in.a2 = a.action[2 * ld + i];
    {
        const char* p = reinterpret_cast<const char*>(a.mults + i);
#pragma unroll
        for (int k = 0; k < 11; ++k, p += row_bytes) in.mm[k] = *reinterpret_cast<const T*>(p);
    }
    in.err_o0 = a.err_o[i]; in.err_o1 = a.err_o[ld + i]; in.err_o2 = a.err_o[2 * ld + i];
    in.ep_return = a.ep_return[i];
    in.episode = a.auto_reset ? a.episode[i] : 0u;
    {
        const char* p = reinterpret_cast<const char*>(a.recent + i);
#pragma unroll
        for (int s = 0; s < 10; ++s) {
#pragma unroll
            for (int c = 0; c < 3; ++c, p += row_bytes) in.ring[s][c] = *reinterpret_cast<const T*>(p);
        }
    }
    if constexpr (STAGE) auv_step_env<T, CYL>(a, i, in, GatherStaged{a.flow, stage});
    else auv_step_env<T, CYL>(a, i, in, GatherDirect<T>{a.flow});
}

template <typename T> struct AuvResetArgs {
    AuvDev<T> P;
    long n, ld;
    T* state; T* obs; int32_t* istep; T* mults; T* target; T* err_o; T* recent; T* ep_return;
    const int32_t* iwp;
    const uint32_t* episode; const uint8_t* mask;
    const T* init;  // nullable [4][ld]: x, y, heading, headingTarget (fixedInitialValues)
    unsigned long long seed, env_id0;
    int apply_noise;
};

// AuvEnv.reset, verySimpleAuv.py:216-262
template <typename T>
__global__ void __launch_bounds__(128)
auv_reset_kernel(const __grid_constant__ AuvResetArgs<T> a) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.n) return;
    if (a.mask != nullptr && a.mask[i] == 0) return;
    const long ld = a.ld;
    T mm[11], x, y, psi, target, offset;
    draw_reset_auv(a.P, a.seed, a.env_id0 + (unsigned long long)i, a.episode ? a.episode[i] : 0u, a.apply_noise != 0, mm, &x, &y, &psi, &target, &offset);
    if (a.init != nullptr) { x = a.init[i]; y = a.init[ld + i]; psi = a.init[2 * ld + i]; target = a.init[3 * ld + i]; }
    T tx = T(0), ty = T(0);
    if (a.P.cyl) { const int w = a.iwp[i]; tx = a.P.wp[w][0]; ty = a.P.wp[w][1]; target = a.P.wp[w][2]; }
#pragma unroll
    for (int k = 0; k < 11; ++k) a.mults[k * ld + i] = mm[k];
    a.state[i] = x; a.state[ld + i] = y; a.state[2 * ld + i] = psi;
    a.state[3 * ld + i] = T(0); a.state[4 * ld + i] = T(0); a.state[5 * ld + i] = T(0);
    a.target[i] = target; a.target[ld + i] = offset;
    a.istep[i] = 0;
    a.ep_return[i] = T(0);
#pragma unroll
    for (int k = 0; k < 30; ++k) a.recent[k * ld + i] = T(0);
    const T herr = angle_error(target, psi);
    a.err_o[i] = tx - x; a.err_o[ld + i] = ty - y; a.err_o[2 * ld + i] = herr;
    T obs[11];
    if (a.P.cyl) observe_auv<true>(tx, ty, x, y, psi, T(0), T(0), T(0), target, tx - x, ty - y, herr, obs);
    else observe_auv<false>(tx, ty, x, y, psi, T(0), T(0), T(0), target, tx - x, ty - y, herr, obs);
#pragma unroll
    for (int k = 0; k < 11; ++k) a.obs[k * ld + i] = obs[k];
}

// stand-alone ReconstructedFlow.interp: t [n], xy [2][ld] -> out [3][ld]
template <typename T>
__global__ void flow_interp_kernel(const FlowDev<T> f, long n, long ld, const T* t, const T* xy, T* out) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (f.nc == 3) {
        T r[3];
        flow_interp<T, 3>(f, t[i], xy[i], xy[ld + i], r);
        out[i] = r[0]; out[ld + i] = r[1]; out[2 * ld + i] = r[2];
    } else {
        T r[2];
        flow_interp<T, 2>(f, t[i], xy[i], xy[ld + i], r);
        out[i] = r[0]; out[ld + i] = r[1];
    }
}

// ReconstructedFlow.scale (flowGenerator.py:80-90) on the field values: base [cells][3] -> out [cells][nc_out]
template <typename T>
__global__ void flow_scale_kernel(long cells, const T* base, T* out, int nc_out, T vel, T turb) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cells) return;
    const T u = (base[3 * i] * vel - vel) * turb + vel;
    const T v = (base[3 * i + 1] * vel - T(0)) * turb;
    out[nc_out * i] = u;
    out[nc_out * i + 1] = v;
    if (nc_out == 3) out[3 * i + 2] = base[3 * i + 2] / tmax(T(1e-6), (vel * turb) * (vel * turb));
}

// ---------------------------------------------------------------------------
// ReconstructedFlow.__init__ (flowGenerator.py:15-23): baseFlowData[t] = Re(modes @ coeffs[:, t]) + lt_mean, written as
// ONE pass in the layout and precision the env reads: out T [nt][P] (P = Ny * Nx * 3 values of a plane), accumulated in
// fp64 like the reference's numpy matmul.  modes [P][K] and coeffs [K][nt] are fp64, complex (interleaved re, im: the
// pySPOD blobs are complex128) or real.
//
// This is the one dense contraction of the code base, so it runs on the tensor cores: fp64 has no tcgen05 / TMEM path, the
// fp64 tensor-core instruction of sm_100 is the warp-level DMMA (mma.sync.m8n8k4.f64).  Only the real part is wanted:
// Re(m c) = mr cr - mi ci is ONE real GEMM of depth 2K over the interleaved storage, A'[p][2k + s] = modes' raw doubles
// and B'[2k + s][t] = (cr, -ci) - half the arithmetic of the complex product a library ZGEMM forms and then discards.
// CTA = 128 (p) x 64 (t) outputs, 8 warps of 32 x 32 (4 x 4 DMMA tiles, 32 fp64 accumulators per thread), depth in steps of
// 16 through shared memory (padded: both fragment loads are conflict-free), next tiles prefetched into registers while the
// current ones are multiplied; mean, conversion to T and the [nt][P] layout are fused into the epilogue - no [P][nt]
// intermediate, no transpose, no separate "+ mean" pass.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void dmma_m8n8k4(double (&d)[2], double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};" : "+d"(d[0]), "+d"(d[1]) : "d"(a), "d"(b));
}

template <typename T>
__global__ void __launch_bounds__(256)
flow_reconstruct_kernel(long P, int K, int nt, const double* __restrict__ modes, int modes_complex, const double* __restrict__ coeffs,
                        int coeffs_complex, const double* __restrict__ mean, T* __restrict__ out) {
    constexpr int BM = 128, BN = 64, BK = 16, LDA = BK + 4, LDB = BN + 8;
    __shared__ double a_s[BM][LDA];    // A'[p][k']: rows 20 doubles apart -> the 8 x 4 fragment read (8 rows x 4 consecutive) hits 32 distinct 8-byte banks
    __shared__ double b_s[BK][LDB];    // B'[k'][t]: rows 72 doubles apart -> the 4 x 8 fragment read likewise
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, tig = lane & 3;
    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 32;     // this warp's 32 x 32 corner inside the CTA tile
    const long p0 = (long)blockIdx.x * BM;
    const int t0 = blockIdx.y * BN;
    const int ms = modes_complex ? 2 : 1, cs = coeffs_complex ? 2 : 1;
    const int depth = (modes_complex && coeffs_complex) ? 2 : 1;   // real depth per mode: (re, im) pairs only when both are complex
    const int KD = K * depth;
    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.;
    // global -> register staging: A' 128 x 16 = 8 doubles per thread (row = tid / 2, 8 consecutive k'), B' 16 x 64 = 4 per thread
    double ra[8], rb[4];
    const int a_row = tid >> 1, a_k = (tid & 1) * 8;
    const int b_k = tid >> 4, b_t = (tid & 15) * 4;
    auto fetch = [&](int k0) {
        const long p = p0 + a_row;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const int kd = k0 + a_k + e;
            const int k = kd / depth, sft = kd - k * depth;
            ra[e] = (p < P && kd < KD) ? modes[(p * K + k) * ms + sft] : 0.;
        }
        const int kd = k0 + b_k;
        const int k = kd / depth, sft = kd - k * depth;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int t = t0 + b_t + e;
            const double v = (t < nt && kd < KD) ? coeffs[((long)k * nt + t) * cs + sft] : 0.;
            rb[e] = sft ? -v : v;                               // Re(m c) = mr cr - mi ci
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < KD; k0 += BK) {
#pragma unroll
        for (int e = 0; e < 8; ++e) a_s[a_row][a_k + e] = ra[e];
#pragma unroll
        for (int e = 0; e < 4; ++e) b_s[b_k][b_t + e] = rb[e];
        __syncthreads();
        if (k0 + BK < KD) fetch(k0 + BK);                       // in flight while the tensor cores work on this tile
#pragma unroll
        for (int kk = 0; kk < BK; kk += 4) {
            double af[4], bf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) af[i] = a_s[wm + 8 * i + g][kk + tig];
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = b_s[kk + tig][wn + 8 * j + g];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) dmma_m8n8k4(acc[i][j], af[i], bf[j]);
        }
        __syncthreads();
    }
    // accumulator fragment: row (p) = g, columns (t) = 2 tig, 2 tig + 1; the 8 g-lanes of a column write 8 consecutive p
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const long p = p0 + wm + 8 * i + g;
        if (p >= P) continue;
        const double mu = mean[p];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int t = t0 + wn + 8 * j + 2 * tig + c;
                if (t < nt) out[(long)t * P + p] = T(acc[i][j][c] + mu);
            }
        }
    }
}

// ---------------------------------------------------------------------------
// CustomReplayBuffer.add (tag_00.../main_02_sbl_contrib_customBuffer.py:57-160): every transition of the
// legacy env is stored together with its mirror images (obs / action sign flips); reward and done are
// unchanged.  Slot (pos + t) % buffer_size holds transformation t of the whole batch, as upstream.
// obs, next_obs T [11][ld], act T [3][ld] (SoA, straight from the env) -> buffers [buffer_size][n][k] (AoS rows,
// the layout a learner samples).  One thread per (environment, transformation).
// ---------------------------------------------------------------------------
__constant__ float kReplaySignObs[5][11] = {
    {1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1}, {-1, -1, 1, 1, -1, -1, -1, -1, 1, 1, 1}, {-1, 1, 1, 1, -1, 1, -1, 1, 1, 1, 1},
    {1, -1, 1, 1, 1, -1, 1, -1, 1, 1, 1}, {1, 1, -1, 1, 1, 1, 1, 1, -1, 1, 1}};
__constant__ float kReplaySignAct[5][3] = {{1, 1, 1}, {-1, -1, 1}, {-1, 1, 1}, {1, -1, 1}, {1, 1, -1}};

template <typename T>
__global__ void replay_add_symmetric_kernel(long n, long ld, const T* obs, const T* next_obs, const T* act, const T* reward,
                                            const uint8_t* done, const uint8_t* timeout, T* b_obs, T* b_next, T* b_act, T* b_rew,
                                            uint8_t* b_done, uint8_t* b_timeout, long buffer_size, long pos, int n_transforms) {
    const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * n_transforms) return;
    const int t = (int)(e / n);
    const long i = e - (long)t * n;
    const long row = ((pos + t) % buffer_size) * n + i;
#pragma unroll
    for (int k = 0; k < 11; ++k) {
        const T sg = T(kReplaySignObs[t][k]);
        b_obs[row * 11 + k] = obs[k * ld + i] * sg;
        b_next[row * 11 + k] = next_obs[k * ld + i] * sg;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) b_act[row * 3 + k] = act[k * ld + i] * T(kReplaySignAct[t][k]);
    b_rew[row] = reward[i];
    b_done[row] = done[i];
    if (b_timeout != nullptr) b_timeout[row] = timeout != nullptr ? timeout[i] : 0;   // main_02...:150-151
}

}  // namespace mvrl
