// C ABI of libmvrl.so (see include/mvrl.h).  Host side: argument checking,
// conversion of the vehicle constants to the compute type, kernel selection
// (dtype x action mode x default-sparsity x fast-math) and launches on the
// caller's stream.  No allocation, no synchronisation per call.
#include <cuda_runtime.h>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "mvrl_host.h"
#include "rov6_kernels.cuh"

using namespace mvrl;

// ---------------------------------------------------------------------------
// error reporting
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";

int mvrl_fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

extern "C" MVRL_API int mvrl_version(void) { return MVRL_VERSION; }
extern "C" MVRL_API const char* mvrl_last_error(void) { return g_err; }
extern "C" MVRL_API int mvrl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ---------------------------------------------------------------------------
// small dense linear algebra for mvrl_rov6_default_params (host, long double)
// ---------------------------------------------------------------------------
bool mvrl_invert_n(const double* a, double* out, int n) {
    long double w[6][12];
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) { w[i][j] = a[i * n + j]; w[i][n + j] = (i == j) ? 1.0L : 0.0L; }
    for (int c = 0; c < n; ++c) {
        int piv = c;
        for (int r = c + 1; r < n; ++r) if (fabsl(w[r][c]) > fabsl(w[piv][c])) piv = r;
        if (fabsl(w[piv][c]) < 1e-300L) return false;
        if (piv != c) for (int j = 0; j < 2 * n; ++j) { long double t = w[c][j]; w[c][j] = w[piv][j]; w[piv][j] = t; }
        const long double d = w[c][c];
        for (int j = 0; j < 2 * n; ++j) w[c][j] /= d;
        for (int r = 0; r < n; ++r) {
            if (r == c) continue;
            const long double f = w[r][c];
            if (f != 0.0L) for (int j = 0; j < 2 * n; ++j) w[r][j] -= f * w[c][j];
        }
    }
    for (int i = 0; i < n; ++i) for (int j = 0; j < n; ++j) out[i * n + j] = (double)w[i][n + j];
    return true;
}

extern "C" MVRL_API int mvrl_rov6_default_params(MvrlRov6Params* p) {
    if (!p) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_default_params: null output");
    memset(p, 0, sizeof(*p));
    const double pi = 3.14159265358979323846;
    // dynamicsModel_BlueROV2_Heavy_6DoF.py:83-184
    p->rho_f = 1000.; p->m = 11.4; p->Length = 0.457;
    p->CG[2] = 0.05;
    p->I[0] = p->I[4] = p->I[8] = 0.16;
    p->Xudot = -5.5; p->Yvdot = -12.7; p->Zwdot = -14.57; p->Kpdot = p->Mqdot = p->Nrdot = -0.12;
    p->Xuu = -18.18; p->Yvv = -21.66; p->Zww = -36.99; p->Kpp = p->Mqq = p->Nrr = -1.55; p->Mww = -1.55;
    p->Xu = -4.03; p->Yv = -6.22; p->Zw = -5.18; p->Kp = p->Mq = p->Nr = -0.07;
    const double dispVol = p->m / p->rho_f;
    p->W = p->m * 9.81;
    p->B = dispVol * p->rho_f * 9.81;
    const double D = 0.1;
    const double Kt = 40. / (1000. * pow(3500. / 60., 2.) * pow(D, 4.));
    p->thrust_coef = p->rho_f * pow(D, 4.) * Kt;
    p->rpm_max = 3500.; p->rpm_deadband = 300.;
    // M = Mrb + Ma with Ma[2][2] = -Zvdot = 0 (6DoF.py:286-299)
    const double m = p->m, xg = p->CG[0], yg = p->CG[1], zg = p->CG[2];
    const double Mrb[36] = {m, 0, 0, 0, m * zg, -m * yg,  0, m, 0, -m * zg, 0, m * xg,  0, 0, m, m * yg, -m * xg, 0,
                            0, -m * zg, m * yg, p->I[0], p->I[1], p->I[2],  m * zg, 0, -m * xg, p->I[3], p->I[4], p->I[5],
                            -m * yg, m * xg, 0, p->I[6], p->I[7], p->I[8]};
    const double Zvdot = 0.;
    const double Ma[6] = {-p->Xudot, -p->Yvdot, -Zvdot, -p->Kpdot, -p->Mqdot, -p->Nrdot};
    for (int i = 0; i < 36; ++i) p->M[i] = Mrb[i];
    for (int i = 0; i < 6; ++i) p->M[i * 6 + i] += Ma[i];
    if (!mvrl_invert_n(p->M, p->Minv, 6)) return mvrl_fail(MVRL_EINVAL, "singular mass matrix");
    // thruster geometry, 6DoF.py:164-212, and allocation, resources.py:19-35
    const double al = 33. / 180. * pi, lx = 0.1475, ly = 0.101, lz = 0.068, lxv = 0.120, lyv = 0.22, lzv = 0.0;
    const double pos[8][3] = {{lx, ly, lz}, {lx, -ly, lz}, {-lx, ly, lz}, {-lx, -ly, lz},
                              {lxv, lyv, lzv}, {lxv, -lyv, lzv}, {-lxv, lyv, lzv}, {-lxv, -lyv, lzv}};
    const double nrm[8][3] = {{cos(al), -sin(al), 0}, {cos(al), sin(al), 0}, {-cos(al), -sin(al), 0}, {-cos(al), sin(al), 0},
                              {0, 0, -1}, {0, 0, 1}, {0, 0, 1}, {0, 0, -1}};
    for (int i = 0; i < 8; ++i) {
        const double* r = pos[i]; const double* n = nrm[i];
        p->A[0 * 8 + i] = n[0]; p->A[1 * 8 + i] = n[1]; p->A[2 * 8 + i] = n[2];
        p->A[3 * 8 + i] = r[1] * n[2] - r[2] * n[1];
        p->A[4 * 8 + i] = r[2] * n[0] - r[0] * n[2];
        p->A[5 * 8 + i] = r[0] * n[1] - r[1] * n[0];
    }
    // A has full row rank: pinv(A) = A^T (A A^T)^-1
    double AAt[36], AAtInv[36];
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) {
        long double s = 0; for (int k = 0; k < 8; ++k) s += (long double)p->A[i * 8 + k] * p->A[j * 8 + k];
        AAt[i * 6 + j] = (double)s;
    }
    if (!mvrl_invert_n(AAt, AAtInv, 6)) return mvrl_fail(MVRL_EINVAL, "rank-deficient allocation matrix");
    for (int i = 0; i < 8; ++i) for (int j = 0; j < 6; ++j) {
        long double s = 0; for (int k = 0; k < 6; ++k) s += (long double)p->A[k * 8 + i] * AAtInv[k * 6 + j];
        p->Ainv[i * 6 + j] = (double)s;
    }
    // PID, 6DoF.py:46-54
    const double wind[6] = {2., 2., 2., 90. / 180. * pi, 90. / 180. * pi, 90. / 180. * pi};
    const double fmx[6] = {50., 50., 50., 1., 1., 2.};
    const double kp[6] = {25., 25., 25., 10., 10., 1.}, ki[6] = {2., 2., 2., 0.1, 0.1, 0.2}, kd[6] = {20., 20., 20., 5., 5., 0.65};
    for (int i = 0; i < 6; ++i) { p->pid_windup[i] = wind[i]; p->pid_max[i] = fmx[i]; p->pid_Kp[i] = kp[i]; p->pid_Ki[i] = ki[i]; p->pid_Kd[i] = kd[i]; }
    p->disable_thrusters = 0;
    return MVRL_OK;
}

// ---------------------------------------------------------------------------
// handle
// ---------------------------------------------------------------------------
struct MvrlRov6 {
    MvrlRov6Params p;
    MvrlRov6Config c;
    bool sp;  // default sparsity pattern holds -> specialised kernels
    bool x2;  // fp32: two environments per thread on the packed FFMA2 path (MVRL_NO_X2=1 in the environment disables it)
    bool constp;  // fp32 constants equal the compiled-in default vehicle bit for bit -> kernels with literal constants (MVRL_NO_CONSTP=1 disables)
    Rov6Dev<float> pf;
    Rov6Dev<double> pd;
    // resources of mvrl_rov6_step_host (created on first use, released by destroy)
    // three queues, one per engine: hs[0] uploads, hs[1] kernels, hs[2] downloads; chunk c flows
    // hs[0] -ev_up[c]-> hs[1] -ev_k[c]-> hs[2], so no engine ever waits behind another one's backlog
    static constexpr int kStreams = 3;
    static constexpr int kMaxChunks = 64;
    cudaStream_t hs[kStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_in = nullptr, ev_out[kStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_up[kMaxChunks] = {}, ev_k[kMaxChunks] = {};
    void* stage_act = nullptr;   // AoS [n][A] copy of the host actions
    void* stage_obs = nullptr;   // AoS [n][9] obs ready for download
    size_t stage_act_bytes = 0, stage_obs_bytes = 0;
    // the whole host step (copies + kernels over all chunks) captured once per distinct set of
    // pointers and replayed with a single cudaGraphLaunch
    static constexpr int kGraphs = 4;
    struct HostGraph { unsigned long long key[20]; cudaGraphExec_t exec; unsigned long long used; };
    HostGraph graphs[kGraphs] = {};
    unsigned long long graph_clock = 0;
};

template <typename T> static void to_dev(const MvrlRov6Params& p, Rov6Dev<T>& d) {
    const double pi = 3.14159265358979323846;
    d.m = T(p.m); d.xg = T(p.CG[0]); d.yg = T(p.CG[1]); d.zg = T(p.CG[2]);
    d.Ixx = T(p.I[0]); d.Iyy = T(p.I[4]); d.Izz = T(p.I[8]); d.Ixy = T(p.I[1]); d.Ixz = T(p.I[2]); d.Iyz = T(p.I[5]);
    d.Xud = T(p.Xudot); d.Yvd = T(p.Yvdot); d.Zwd = T(p.Zwdot); d.Kpd = T(p.Kpdot); d.Mqd = T(p.Mqdot); d.Nrd = T(p.Nrdot);
    d.Xu = T(p.Xu); d.Yv = T(p.Yv); d.Yp = T(p.Yp); d.Yr = T(p.Yr); d.Zw = T(p.Zw); d.Zq = T(p.Zq); d.Kv = T(p.Kv);
    d.Kp = T(p.Kp); d.Kr = T(p.Kr); d.Mw = T(p.Mw); d.Mq = T(p.Mq); d.Nv = T(p.Nv); d.Np = T(p.Np); d.Nr = T(p.Nr);
    d.Xuu = T(p.Xuu); d.Yvv = T(p.Yvv); d.Ypp = T(p.Ypp); d.Yrr = T(p.Yrr); d.Zww = T(p.Zww); d.Zqq = T(p.Zqq); d.Kvv = T(p.Kvv);
    d.Kpp = T(p.Kpp); d.Krr = T(p.Krr); d.Mww = T(p.Mww); d.Mqq = T(p.Mqq); d.Nvv = T(p.Nvv); d.Npp = T(p.Npp); d.Nrr = T(p.Nrr);
    d.WmB = T(p.W - p.B);
    d.gx = T(p.CG[0] * p.W - p.CB[0] * p.B); d.gy = T(p.CG[1] * p.W - p.CB[1] * p.B); d.gz = T(p.CG[2] * p.W - p.CB[2] * p.B);
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 8; ++j) d.A[i][j] = T(p.A[i * 8 + j]);
    for (int i = 0; i < 8; ++i) for (int j = 0; j < 6; ++j) d.Ainv[i][j] = T(p.Ainv[i * 6 + j]);
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) d.Minv[i][j] = T(p.Minv[i * 6 + j]);
    d.thrust_k = T(p.thrust_coef / 3600.);
    d.inv_thrust_coef = T(1. / p.thrust_coef);
    d.rpm_max = T(p.rpm_max); d.rpm_db = T(p.rpm_deadband);
    d.f_max = T(p.thrust_coef * (p.rpm_max / 60.) * (p.rpm_max / 60.));
    d.f_db = T(p.thrust_coef * (p.rpm_deadband / 60.) * (p.rpm_deadband / 60.));
    for (int i = 0; i < 6; ++i) {
        d.pKp[i] = T(p.pid_Kp[i]); d.pKi[i] = T(p.pid_Ki[i]); d.pKd[i] = T(p.pid_Kd[i]);
        d.pWind[i] = T(p.pid_windup[i]); d.pMax[i] = T(p.pid_max[i]);
    }
    d.inv_3L = T(1. / (p.Length * 3.)); d.act_pos = T(2. * p.Length);
    d.act_ang = T(45. / 180. * pi); d.inv_ang = T(1. / (45. / 180. * pi));
    d.mX = T(p.m - p.Xudot); d.mY = T(p.m - p.Yvdot); d.mZ = T(p.m - p.Zwdot); d.mzg = T(p.m * p.CG[2]);
    d.cVW = T(p.Yvdot - p.Zwdot); d.cUW = T(p.Zwdot - p.Xudot); d.cUV = T(p.Xudot - p.Yvdot);
    d.cQR = T(p.I[8] - p.I[4] + p.Mqdot - p.Nrdot); d.cPR = T(p.I[0] - p.I[8] + p.Nrdot - p.Kpdot);
    d.cPQ = T(p.I[4] - p.I[0] + p.Kpdot - p.Mqdot);
    d.thrusters_on = p.disable_thrusters ? 0 : 1;
}

// Does the parameter set have the reference's default sparsity?  (Tiny pinv /
// inverse round-off entries count as zero; they are < 1e-13 of the scale.)
static bool default_sparsity(const MvrlRov6Params& p) {
    auto z = [](double v, double scale) { return fabs(v) <= 1e-13 * scale; };
    if (p.CG[0] != 0 || p.CG[1] != 0 || p.CB[0] != 0 || p.CB[1] != 0) return false;
    if (p.I[1] != 0 || p.I[2] != 0 || p.I[5] != 0 || p.I[3] != 0 || p.I[6] != 0 || p.I[7] != 0) return false;
    if (p.W - p.B != 0) return false;
    if (p.Yp != 0 || p.Yr != 0 || p.Zq != 0 || p.Kv != 0 || p.Kr != 0 || p.Mw != 0 || p.Nv != 0 || p.Np != 0) return false;
    if (p.Ypp != 0 || p.Yrr != 0 || p.Zqq != 0 || p.Kvv != 0 || p.Krr != 0 || p.Nvv != 0 || p.Npp != 0) return false;
    double amax = 0, imax = 0, mmax = 0;
    for (int i = 0; i < 48; ++i) { amax = fmax(amax, fabs(p.A[i])); imax = fmax(imax, fabs(p.Ainv[i])); }
    for (int i = 0; i < 36; ++i) mmax = fmax(mmax, fabs(p.Minv[i]));
    for (int j = 0; j < 8; ++j) {
        const bool horiz = j < 4;
        if (horiz ? !z(p.A[2 * 8 + j], amax) : !(z(p.A[0 * 8 + j], amax) && z(p.A[1 * 8 + j], amax) && z(p.A[5 * 8 + j], amax))) return false;
        if (horiz ? !(z(p.Ainv[j * 6 + 2], imax) && z(p.Ainv[j * 6 + 3], imax) && z(p.Ainv[j * 6 + 4], imax)) : !z(p.Ainv[j * 6 + 5], imax)) return false;
    }
    for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) {
        const bool keep = (i == j) || (i == 0 && j == 4) || (i == 4 && j == 0) || (i == 1 && j == 3) || (i == 3 && j == 1);
        if (!keep && !z(p.Minv[i * 6 + j], mmax)) return false;
    }
    return true;
}

// the default vehicle as compiled into the CONSTP kernels, and the flat view both sides are compared through
static const Rov6Dev<float> kRov6DefaultF32 = MVRL_ROV6_DEFAULT_INIT_F32;
static constexpr size_t kRov6DevWords = offsetof(Rov6Dev<float>, thrusters_on) / sizeof(float);
static_assert(kRov6DevWords == MVRL_ROV6_DEFAULT_WORDS, "rov6_default_consts.h is out of date: run tools/gen_default_consts.py");

// Flattened fp32 device constants of a parameter set (what tools/gen_default_consts.py writes into rov6_default_consts.h)
extern "C" MVRL_API int mvrl_rov6_dev_constants_f32(const MvrlRov6Params* params, float* out, int capacity) {
    if (!params || !out || capacity < (int)kRov6DevWords) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_dev_constants_f32: need room for %d floats", (int)kRov6DevWords);
    Rov6Dev<float> d;
    memset(&d, 0, sizeof(d));
    to_dev(*params, d);
    memcpy(out, &d, kRov6DevWords * sizeof(float));
    return (int)kRov6DevWords;
}

extern "C" MVRL_API int mvrl_rov6_create(MvrlRov6** out, const MvrlRov6Params* params, const MvrlRov6Config* cfg) {
    if (!out || !params || !cfg) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_create: null argument");
    if (cfg->dtype != MVRL_F32 && cfg->dtype != MVRL_F64) return mvrl_fail(MVRL_EINVAL, "dtype must be MVRL_F32 or MVRL_F64");
    if (cfg->action_mode < 0 || cfg->action_mode > 2) return mvrl_fail(MVRL_EINVAL, "bad action_mode %d", cfg->action_mode);
    if (cfg->n_sub < 1) return mvrl_fail(MVRL_EINVAL, "n_sub must be >= 1");
    if (!(cfg->dt > 0)) return mvrl_fail(MVRL_EINVAL, "dt must be > 0");
    if (!(params->thrust_coef > 0)) return mvrl_fail(MVRL_EINVAL, "thrust_coef must be > 0");
    { const int rc = mvrl_require_device(cfg->device); if (rc != MVRL_OK) return rc; }
    MvrlRov6* h = new (std::nothrow) MvrlRov6();
    if (!h) return mvrl_fail(MVRL_EINVAL, "out of host memory");
    h->p = *params;
    h->c = *cfg;
    h->sp = default_sparsity(*params);
    { const char* e = getenv("MVRL_NO_X2"); h->x2 = !(e && e[0] == '1'); }
    memset(&h->pf, 0, sizeof(h->pf));
    memset(&h->pd, 0, sizeof(h->pd));
    to_dev(*params, h->pf);
    to_dev(*params, h->pd);
    { const char* e = getenv("MVRL_NO_CONSTP");
      h->constp = !(e && e[0] == '1') && h->sp && h->pf.thrusters_on == 1 && memcmp(&h->pf, &kRov6DefaultF32, kRov6DevWords * sizeof(float)) == 0; }
    *out = h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_rov6_destroy(MvrlRov6* h) {
    if (!h) return MVRL_OK;
    if (h->hs[0] || h->stage_act || h->stage_obs) {
        MvrlDeviceGuard guard(h->c.device);
        for (int i = 0; i < MvrlRov6::kStreams; ++i) {
            if (h->hs[i]) cudaStreamDestroy(h->hs[i]);
            if (h->ev_out[i]) cudaEventDestroy(h->ev_out[i]);
        }
        if (h->ev_in) cudaEventDestroy(h->ev_in);
        for (int i = 0; i < MvrlRov6::kMaxChunks; ++i) {
            if (h->ev_up[i]) cudaEventDestroy(h->ev_up[i]);
            if (h->ev_k[i]) cudaEventDestroy(h->ev_k[i]);
        }
        for (int i = 0; i < MvrlRov6::kGraphs; ++i) if (h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
        cudaFree(h->stage_act);
        cudaFree(h->stage_obs);
    }
    delete h;
    return MVRL_OK;
}
extern "C" MVRL_API int mvrl_rov6_is_specialised(const MvrlRov6* h) { return (h && h->sp) ? (h->constp ? 2 : 1) : 0; }

#define grid_for mvrl_grid_for
#define check_launch mvrl_check_launch

int mvrl_require_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return mvrl_fail(MVRL_ENODEV, "no CUDA device: libmvrl has no CPU path");
    }
    if (device < 0 || device >= ndev) return mvrl_fail(MVRL_EINVAL, "device %d out of range (%d devices)", device, ndev);
    return MVRL_OK;
}

// ---------------------------------------------------------------------------
// step
// ---------------------------------------------------------------------------
// Two fp32 environments per thread (packed FFMA2 path) need 8-byte aligned rows.
template <typename T> static bool x2_layout_ok(const Rov6StepArgs<T>& a) {
    if (sizeof(T) != 4 || (a.ld & 1)) return false;
    const void* ptrs[] = {a.state, a.action, a.obs, a.reward, a.setpoint, a.path, a.ctrl, a.istep, a.episode};
    for (const void* p : ptrs) if (((uintptr_t)p) & 7u) return false;
    if (((uintptr_t)a.done) & 1u) return false;   // the two done flags of a thread go out as one 2-byte store
    return true;
}

// x2: two environments per thread; constp: the default vehicle, constants as literals
template <typename T, int MODE, bool SP, bool FAST>
static void launch_step(const Rov6StepArgs<T>& a, bool x2, bool constp, cudaStream_t s) {
    if constexpr (sizeof(T) == 4) {
        if (x2 && x2_layout_ok(a)) {
            const int64_t threads = (a.n + 1) / 2;
            // rpm mode keeps its constants on the argument: literals make it no faster at 168 registers (its few constants
            // sit in uniform registers anyway); they only let the kernel fit 128 registers without spilling (16 warps per SM)
            if constexpr (SP && !FAST && MODE != ACT_RPM) {
                if (constp) {
                    rov6_step_kernel<F2, MODE, SP, FAST, true><<<grid_for(threads, StepLaunch<F2>::BLOCK), StepLaunch<F2>::BLOCK, 0, s>>>(a);
                    return;
                }
            }
            rov6_step_kernel<F2, MODE, SP, FAST><<<grid_for(threads, StepLaunch<F2>::BLOCK), StepLaunch<F2>::BLOCK, 0, s>>>(a);
            return;
        }
    }
    rov6_step_kernel<T, MODE, SP, FAST><<<grid_for(a.n, StepLaunch<T>::BLOCK), StepLaunch<T>::BLOCK, 0, s>>>(a);
}
template <typename T, bool FAST>
static void dispatch_step(const Rov6StepArgs<T>& a, int mode, bool sp, bool x2, bool constp, cudaStream_t s) {
    switch (mode * 2 + (sp ? 1 : 0)) {
        case 0: launch_step<T, ACT_RPM, false, FAST>(a, x2, constp, s); break;
        case 1: launch_step<T, ACT_RPM, true, FAST>(a, x2, constp, s); break;
        case 2: launch_step<T, ACT_FORCE, false, FAST>(a, x2, constp, s); break;
        case 3: launch_step<T, ACT_FORCE, true, FAST>(a, x2, constp, s); break;
        case 4: launch_step<T, ACT_SETPOINT, false, FAST>(a, x2, constp, s); break;
        default: launch_step<T, ACT_SETPOINT, true, FAST>(a, x2, constp, s); break;
    }
}

template <typename T>
static void fill_step_args(const MvrlRov6* h, const Rov6Dev<T>& P, int64_t first, int64_t n, int64_t ld, const MvrlRov6Buffers* b, Rov6StepArgs<T>& a) {
    auto off = [first](void* p) -> T* { return p ? (T*)p + first : nullptr; };
    a.P = P; a.n = n; a.ld = ld;
    a.state = off(b->state); a.action = off(b->action); a.obs = off(b->obs); a.reward = off(b->reward);
    a.done = b->done + first; a.istep = b->istep + first; a.setpoint = off(b->setpoint); a.path = off(b->path); a.ctrl = off(b->ctrl);
    a.episode = b->episode ? b->episode + first : nullptr; a.term_obs = off(b->terminal_obs); a.aux = off(b->aux); a.stats = b->ep_stats;
    a.dt = T(h->c.dt); a.h = T(h->c.dt / h->c.n_sub);
    a.hh = T(0.5) * a.h; a.h6 = a.h / T(6); a.h3 = a.h / T(3);   // in T arithmetic, like the kernel used to
    const T dtc[2] = {T(0), a.hh};
    for (int i = 0; i < 2; ++i) {
        a.pid_inv_dt[i] = T(1) / (dtc[i] > T(1e-9) ? dtc[i] : T(1e-9)); a.pid_half_dt[i] = T(0.5) * dtc[i];
        for (int k = 0; k < 6; ++k) a.pid_kd_inv_dt[i][k] = P.pKd[k] * a.pid_inv_dt[i];
    }
    a.n_sub = h->c.n_sub; a.max_steps = h->c.max_steps;
    a.seed = h->c.seed; a.env_id0 = h->c.env_id0 + (unsigned long long)first;
    a.auto_reset = h->c.auto_reset; a.fixed_sp = h->c.fixed_sp;
}

static int check_step_args(const MvrlRov6* h, int64_t first, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const char* who) {
    if (!h || !b) return mvrl_fail(MVRL_EINVAL, "%s: null argument", who);
    if (first < 0 || n < 0 || ld < first + n) return mvrl_fail(MVRL_EINVAL, "%s: need 0 <= first, 0 <= n, first + n <= ld (first=%lld n=%lld ld=%lld)", who, (long long)first, (long long)n, (long long)ld);
    if (!b->state || !b->action || !b->obs || !b->reward || !b->done || !b->istep || !b->setpoint || !b->path)
        return mvrl_fail(MVRL_EINVAL, "%s: state/action/obs/reward/done/istep/setpoint/path are required", who);
    if (h->c.action_mode == MVRL_ACT_SETPOINT && !b->ctrl) return mvrl_fail(MVRL_EINVAL, "%s: ctrl is required in set-point mode", who);
    if (h->c.auto_reset && !b->episode) return mvrl_fail(MVRL_EINVAL, "%s: episode is required with auto_reset", who);
    return MVRL_OK;
}

// launches the fused step for environments [first, first + n) on stream s
static void launch_step_range(const MvrlRov6* h, int64_t first, int64_t n, int64_t ld, const MvrlRov6Buffers* b, cudaStream_t s) {
    if (h->c.dtype == MVRL_F64) {
        Rov6StepArgs<double> a; fill_step_args(h, h->pd, first, n, ld, b, a);
        dispatch_step<double, false>(a, h->c.action_mode, h->sp, false, false, s);
    } else {
        Rov6StepArgs<float> a; fill_step_args(h, h->pf, first, n, ld, b, a);
        if (h->c.fast_math) dispatch_step<float, true>(a, h->c.action_mode, h->sp, h->x2, h->constp, s);
        else dispatch_step<float, false>(a, h->c.action_mode, h->sp, h->x2, h->constp, s);
    }
}

extern "C" MVRL_API int mvrl_rov6_step(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, mvrl_stream_t stream) {
    { const int rc = check_step_args(h, 0, n, ld, b, "mvrl_rov6_step"); if (rc != MVRL_OK) return rc; }
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    launch_step_range(h, 0, n, ld, b, (cudaStream_t)stream);
    return check_launch("rov6_step");
}

extern "C" MVRL_API int mvrl_rov6_step_range(MvrlRov6* h, int64_t first, int64_t n, int64_t ld, const MvrlRov6Buffers* b, mvrl_stream_t stream) {
    { const int rc = check_step_args(h, first, n, ld, b, "mvrl_rov6_step_range"); if (rc != MVRL_OK) return rc; }
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    launch_step_range(h, first, n, ld, b, (cudaStream_t)stream);
    return check_launch("rov6_step_range");
}

// ---------------------------------------------------------------------------
// step with HOST buffers: chunked upload / transpose / step / transpose / download pipeline
// ---------------------------------------------------------------------------
// AoS [n][K] (row = environment, the layout a host-side VecEnv caller holds) <-> SoA [K][ld].
// Tiles of 32 environments go through shared memory so that both sides are coalesced.
template <typename T, int K>
__global__ void __launch_bounds__(256) aos_to_soa_kernel(long n, long ld, const T* __restrict__ aos, T* __restrict__ soa) {
    constexpr int KP = K | 1;  // odd row pitch: conflict-free column reads
    __shared__ T tile[256 * KP];
    const long base = (long)blockIdx.x * 256;
    const int cnt = (int)((n - base) < 256 ? (n - base) : 256);
    for (int e = threadIdx.x; e < cnt * K; e += 256) tile[(e / K) * KP + (e % K)] = aos[base * K + e];
    __syncthreads();
    if ((int)threadIdx.x < cnt) {
#pragma unroll
        for (int k = 0; k < K; ++k) soa[k * ld + base + threadIdx.x] = tile[threadIdx.x * KP + k];
    }
}

// reward_map / done_map (nullable): device aliases of PINNED host arrays.  The block also forwards its 256 rewards
// and done flags straight to the host (posted PCIe writes, 5 B per environment) so that the download engine has ONE
// copy per piece to do instead of three - each queued copy costs it ~4.5 us (r1k measurements: 13-15 us per piece).
template <typename T, int K>
__global__ void __launch_bounds__(256) soa_to_aos_kernel(long n, long ld, const T* __restrict__ soa, T* __restrict__ aos,
                                                         const T* __restrict__ reward, const uint8_t* __restrict__ done,
                                                         T* __restrict__ reward_map, uint8_t* __restrict__ done_map) {
    constexpr int KP = K | 1;
    __shared__ T tile[256 * KP];
    const long base = (long)blockIdx.x * 256;
    const int cnt = (int)((n - base) < 256 ? (n - base) : 256);
    if ((int)threadIdx.x < cnt) {
#pragma unroll
        for (int k = 0; k < K; ++k) tile[threadIdx.x * KP + k] = soa[k * ld + base + threadIdx.x];
        if (reward_map != nullptr) reward_map[base + threadIdx.x] = reward[base + threadIdx.x];
        if (done_map != nullptr) done_map[base + threadIdx.x] = done[base + threadIdx.x];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < cnt * K; e += 256) aos[base * K + e] = tile[(e / K) * KP + (e % K)];
}

template <typename T>
static void launch_transposes_in(int n_act, long n, long ld, const T* aos, T* soa, cudaStream_t s) {
    const unsigned g = grid_for(n, 256);
    if (n_act == 8) aos_to_soa_kernel<T, 8><<<g, 256, 0, s>>>(n, ld, aos, soa);
    else aos_to_soa_kernel<T, 6><<<g, 256, 0, s>>>(n, ld, aos, soa);
}

static int ensure_host_pipeline(MvrlRov6* h, size_t act_bytes, size_t obs_bytes) {
    if (!h->hs[0]) {
        for (int i = 0; i < MvrlRov6::kStreams; ++i) {
            MVRL_CUDA(cudaStreamCreateWithFlags(&h->hs[i], cudaStreamNonBlocking));
            MVRL_CUDA(cudaEventCreateWithFlags(&h->ev_out[i], cudaEventDisableTiming));
        }
        MVRL_CUDA(cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming));
        for (int i = 0; i < MvrlRov6::kMaxChunks; ++i) {
            MVRL_CUDA(cudaEventCreateWithFlags(&h->ev_up[i], cudaEventDisableTiming));
            MVRL_CUDA(cudaEventCreateWithFlags(&h->ev_k[i], cudaEventDisableTiming));
        }
    }
    if (h->stage_act_bytes < act_bytes) {
        if (h->stage_act) MVRL_CUDA(cudaFree(h->stage_act));
        h->stage_act = nullptr; h->stage_act_bytes = 0;
        MVRL_CUDA(cudaMalloc(&h->stage_act, act_bytes));
        h->stage_act_bytes = act_bytes;
    }
    if (h->stage_obs_bytes < obs_bytes) {
        if (h->stage_obs) MVRL_CUDA(cudaFree(h->stage_obs));
        h->stage_obs = nullptr; h->stage_obs_bytes = 0;
        MVRL_CUDA(cudaMalloc(&h->stage_obs, obs_bytes));
        h->stage_obs_bytes = obs_bytes;
    }
    return MVRL_OK;
}

static void drop_host_graphs(MvrlRov6* h) {
    for (int i = 0; i < MvrlRov6::kGraphs; ++i) {
        if (h->graphs[i].exec) cudaGraphExecDestroy(h->graphs[i].exec);
        h->graphs[i] = MvrlRov6::HostGraph{};
    }
}

// Piece boundaries of the host pipeline: `chunks` equal pieces (0: kDefaultChunks for large batches), multiples of the 256-environment
// transpose tile.  Measured on B200 / PCIe gen5 (r1o, r1p): 4 pieces 0.90e9, 6 0.99e9, 8 1.02e9, 12 1.01e9, 16 0.95e9
// env-steps/s; geometric ramps (small first piece, growing later ones) were all slower than 8 equal pieces, and so were tapered
// plans with a smaller first AND last piece (r2y: 9-12 pieces, end pieces 0.25-0.5 of the others: 0.94-1.08e9 vs 1.085e9).
static constexpr int kDefaultChunks = 8;
static int host_chunk_plan(int64_t n, int chunks, int64_t* first /* [kMaxChunks + 1] */) {
    if (chunks <= 0) {   // default: 8 pieces, but none smaller than 64 Ki environments (a piece costs ~6 us of fixed overhead)
        const int64_t by_size = n / 65536;
        chunks = by_size < 1 ? 1 : (by_size < kDefaultChunks ? (int)by_size : kDefaultChunks);
    }
    const int64_t per = ((n + chunks - 1) / chunks + 255) / 256 * 256;
    int c = 0;
    first[0] = 0;
    while (first[c] < n && c < MvrlRov6::kMaxChunks) { first[c + 1] = (first[c] + per < n) ? first[c] + per : n; ++c; }
    first[c] = n;
    return c;
}

extern "C" MVRL_API int mvrl_host_chunk_count(int64_t n, int chunks) {
    if (n <= 0) return 0;
    int64_t bounds[MvrlRov6::kMaxChunks + 1];
    if (chunks < 0) chunks = -chunks;
    if (chunks > MvrlRov6::kMaxChunks) chunks = MvrlRov6::kMaxChunks;
    return host_chunk_plan(n, chunks, bounds);
}

// device-side alias of a pinned host allocation, or null (pageable memory, null pointer)
static void* mapped_alias(void* host) {
    if (!host) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) return nullptr;
    return at.devicePointer;
}

// queues the chunked pipeline: everything is ordered after `root` and joined back into `root`
static int enqueue_host_step(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const void* actions_host, void* obs_host,
                             void* reward_host, uint8_t* done_host, int chunks, cudaStream_t root) {
    const size_t es = h->c.dtype == MVRL_F64 ? 8 : 4;
    const int n_act = h->c.action_mode == MVRL_ACT_RPM ? 8 : 6;
    int64_t bounds[MvrlRov6::kMaxChunks + 1];
    const int n_chunks = host_chunk_plan(n, chunks, bounds);
    // done: written by the transpose kernel through the device alias of the host array when it is pinned
    // (cudaHostAlloc / cudaHostRegister, e.g. torch pin_memory); a pageable array keeps the copy-engine path.
    // reward: identically zero for this env (6DoF.py:575), so it does not travel at all - mvrl_rov6_step_host fills the
    // host array with zeros on the host side (once per captured pipeline) instead of shipping 4 B per environment
    // over PCIe every step.
    void* reward_map = nullptr;
    reward_host = nullptr;
    uint8_t* done_map = (uint8_t*)mapped_alias(done_host);
    MVRL_CUDA(cudaEventRecord(h->ev_in, root));
    for (int i = 0; i < MvrlRov6::kStreams; ++i) MVRL_CUDA(cudaStreamWaitEvent(h->hs[i], h->ev_in, 0));
    cudaStream_t s_up = h->hs[0], s_k = h->hs[1], s_dn = h->hs[2];
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t first = bounds[c], cnt = bounds[c + 1] - bounds[c];
        char* d_act = (char*)h->stage_act + (size_t)first * n_act * es;
        char* d_obs = (char*)h->stage_obs + (size_t)first * 9 * es;
        MVRL_CUDA(cudaMemcpyAsync(d_act, (const char*)actions_host + (size_t)first * n_act * es, (size_t)cnt * n_act * es, cudaMemcpyHostToDevice, s_up));
        MVRL_CUDA(cudaEventRecord(h->ev_up[c], s_up));
        MVRL_CUDA(cudaStreamWaitEvent(s_k, h->ev_up[c], 0));
        if (es == 8) launch_transposes_in<double>(n_act, cnt, ld, (const double*)d_act, (double*)b->action + first, s_k);
        else launch_transposes_in<float>(n_act, cnt, ld, (const float*)d_act, (float*)b->action + first, s_k);
        launch_step_range(h, first, cnt, ld, b, s_k);
        if (es == 8) soa_to_aos_kernel<double, 9><<<grid_for(cnt, 256), 256, 0, s_k>>>(cnt, ld, (const double*)b->obs + first, (double*)d_obs,
            (const double*)b->reward + first, b->done + first, reward_map ? (double*)reward_map + first : nullptr, done_map ? done_map + first : nullptr);
        else soa_to_aos_kernel<float, 9><<<grid_for(cnt, 256), 256, 0, s_k>>>(cnt, ld, (const float*)b->obs + first, (float*)d_obs,
            (const float*)b->reward + first, b->done + first, reward_map ? (float*)reward_map + first : nullptr, done_map ? done_map + first : nullptr);
        MVRL_CUDA(cudaEventRecord(h->ev_k[c], s_k));
        MVRL_CUDA(cudaStreamWaitEvent(s_dn, h->ev_k[c], 0));
        MVRL_CUDA(cudaMemcpyAsync((char*)obs_host + (size_t)first * 9 * es, d_obs, (size_t)cnt * 9 * es, cudaMemcpyDeviceToHost, s_dn));
        if (reward_host && !reward_map) MVRL_CUDA(cudaMemcpyAsync((char*)reward_host + (size_t)first * es, (const char*)b->reward + (size_t)first * es, (size_t)cnt * es, cudaMemcpyDeviceToHost, s_dn));
        if (done_host && !done_map) MVRL_CUDA(cudaMemcpyAsync(done_host + first, b->done + first, (size_t)cnt, cudaMemcpyDeviceToHost, s_dn));
    }
    { const int rc = check_launch("rov6_step_host"); if (rc != MVRL_OK) return rc; }
    for (int i = 0; i < MvrlRov6::kStreams; ++i) {
        MVRL_CUDA(cudaEventRecord(h->ev_out[i], h->hs[i]));
        MVRL_CUDA(cudaStreamWaitEvent(root, h->ev_out[i], 0));
    }
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_rov6_step_host(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const void* actions_host,
                                            void* obs_host, void* reward_host, uint8_t* done_host, int chunks, mvrl_stream_t stream) {
    { const int rc = check_step_args(h, 0, n, ld, b, "mvrl_rov6_step_host"); if (rc != MVRL_OK) return rc; }
    if (n == 0) return MVRL_OK;   // an empty batch has no host arrays to name
    if (!actions_host || !obs_host) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_step_host: actions_host and obs_host are required");
    MVRL_ON_DEVICE(h->c.device);
    const size_t es = h->c.dtype == MVRL_F64 ? 8 : 4;
    const int n_act = h->c.action_mode == MVRL_ACT_RPM ? 8 : 6;
    const size_t need_act = (size_t)n * n_act * es, need_obs = (size_t)n * 9 * es;
    if (h->stage_act_bytes < need_act || h->stage_obs_bytes < need_obs) drop_host_graphs(h);  // they hold the old staging pointers
    { const int rc = ensure_host_pipeline(h, need_act, need_obs); if (rc != MVRL_OK) return rc; }
    const bool graph_mode = chunks >= 0;   // chunks < 0: |chunks| pieces queued directly on the streams (no graph)
    if (chunks < 0) chunks = -chunks;
    if (chunks > MvrlRov6::kMaxChunks) chunks = MvrlRov6::kMaxChunks;
    cudaStream_t user = (cudaStream_t)stream;
    const bool zero_reward_now = reward_host != nullptr;   // direct mode: every call; graph mode: when the pipeline is captured
    if (!graph_mode) {
        if (zero_reward_now) memset(reward_host, 0, (size_t)n * es);
        { const int rc = enqueue_host_step(h, n, ld, b, actions_host, obs_host, reward_host, done_host, chunks, user); if (rc != MVRL_OK) return rc; }
        MVRL_CUDA(cudaStreamSynchronize(user));
        return MVRL_OK;
    }
    // everything a captured graph bakes in
    unsigned long long key[20] = {(unsigned long long)n, (unsigned long long)ld, (unsigned long long)chunks,
        (unsigned long long)actions_host, (unsigned long long)obs_host, (unsigned long long)reward_host, (unsigned long long)done_host,
        (unsigned long long)b->state, (unsigned long long)b->action, (unsigned long long)b->obs, (unsigned long long)b->reward,
        (unsigned long long)b->done, (unsigned long long)b->istep, (unsigned long long)b->setpoint, (unsigned long long)b->path,
        (unsigned long long)b->ctrl, (unsigned long long)b->episode, (unsigned long long)b->terminal_obs, (unsigned long long)b->aux,
        (unsigned long long)b->ep_stats};
    MvrlRov6::HostGraph* g = nullptr;
    MvrlRov6::HostGraph* lru = &h->graphs[0];
    for (int i = 0; i < MvrlRov6::kGraphs; ++i) {
        MvrlRov6::HostGraph* e = &h->graphs[i];
        if (e->exec && memcmp(e->key, key, sizeof(key)) == 0) { g = e; break; }
        if (e->used < lru->used) lru = e;
    }
    if (!g) {
        if (zero_reward_now) memset(reward_host, 0, (size_t)n * es);   // the caller's array, zero like every reward of this env
        g = lru;
        if (g->exec) { cudaGraphExecDestroy(g->exec); g->exec = nullptr; }
        cudaGraph_t graph = nullptr;
        MVRL_CUDA(cudaStreamBeginCapture(h->hs[0], cudaStreamCaptureModeThreadLocal));
        // hs[0] is the capture origin: the other streams fork from it and join back
        int rc = MVRL_OK;
        {
            // temporarily treat hs[0] as `root`; chunk streams are hs[1..] plus hs[0] itself
            rc = enqueue_host_step(h, n, ld, b, actions_host, obs_host, reward_host, done_host, chunks, h->hs[0]);
        }
        cudaError_t ce = cudaStreamEndCapture(h->hs[0], &graph);
        if (rc != MVRL_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (ce != cudaSuccess) return mvrl_fail(MVRL_ECUDA, "cudaStreamEndCapture failed: %s", cudaGetErrorString(ce));
        ce = cudaGraphInstantiate(&g->exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ce != cudaSuccess) { g->exec = nullptr; return mvrl_fail(MVRL_ECUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(ce)); }
        memcpy(g->key, key, sizeof(key));
    }
    g->used = ++h->graph_clock;
    MVRL_CUDA(cudaGraphLaunch(g->exec, user));
    MVRL_CUDA(cudaStreamSynchronize(user));   // the host buffers are valid when this returns
    return MVRL_OK;
}

// ---------------------------------------------------------------------------
// derivs
// ---------------------------------------------------------------------------
template <typename T>
static int derivs_impl(const MvrlRov6* h, const Rov6Dev<T>& P, int64_t n, int64_t ld, const void* state, const void* act, const void* t,
                       const void* setpoint, void* ctrl, void* dstate, void* aux, cudaStream_t s) {
    Rov6DerivArgs<T> a;
    a.P = P; a.n = n; a.ld = ld; a.state = (const T*)state; a.act = (const T*)act; a.t = (const T*)t;
    a.setpoint = (const T*)setpoint; a.ctrl = (T*)ctrl; a.dstate = (T*)dstate; a.aux = (T*)aux;
    const unsigned g = grid_for(n, 128);
    switch (h->c.action_mode * 2 + (h->sp ? 1 : 0)) {
        case 0: rov6_derivs_kernel<T, ACT_RPM, false><<<g, 128, 0, s>>>(a); break;
        case 1: rov6_derivs_kernel<T, ACT_RPM, true><<<g, 128, 0, s>>>(a); break;
        case 2: rov6_derivs_kernel<T, ACT_FORCE, false><<<g, 128, 0, s>>>(a); break;
        case 3: rov6_derivs_kernel<T, ACT_FORCE, true><<<g, 128, 0, s>>>(a); break;
        case 4: rov6_derivs_kernel<T, ACT_SETPOINT, false><<<g, 128, 0, s>>>(a); break;
        default: rov6_derivs_kernel<T, ACT_SETPOINT, true><<<g, 128, 0, s>>>(a); break;
    }
    return check_launch("rov6_derivs");
}

extern "C" MVRL_API int mvrl_rov6_derivs(MvrlRov6* h, int64_t n, int64_t ld, const void* state, const void* act, const void* t,
                                const void* setpoint, void* ctrl, void* dstate, void* aux, mvrl_stream_t stream) {
    if (!h || !state || !dstate) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_derivs: null argument");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_derivs: need 0 <= n <= ld");
    if (h->c.action_mode == MVRL_ACT_SETPOINT) {
        if (!t || !setpoint || !ctrl) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_derivs: t, setpoint and ctrl are required in set-point mode");
    } else if (!act) {
        return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_derivs: act is required");
    }
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    cudaStream_t s = (cudaStream_t)stream;
    if (h->c.dtype == MVRL_F64) return derivs_impl<double>(h, h->pd, n, ld, state, act, t, setpoint, ctrl, dstate, aux, s);
    return derivs_impl<float>(h, h->pf, n, ld, state, act, t, setpoint, ctrl, dstate, aux, s);
}

// ---------------------------------------------------------------------------
// reset / pid
// ---------------------------------------------------------------------------
template <typename T>
static int reset_impl(const MvrlRov6* h, const Rov6Dev<T>& P, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const uint8_t* mask,
                      const double* init_sp, cudaStream_t s) {
    Rov6ResetArgs<T> a;
    a.P = P; a.n = n; a.ld = ld;
    a.state = (T*)b->state; a.obs = (T*)b->obs; a.istep = b->istep; a.setpoint = (T*)b->setpoint; a.path = (T*)b->path;
    a.ctrl = (T*)b->ctrl; a.episode = b->episode; a.aux = (T*)b->aux; a.mask = mask;
    a.has_init_sp = init_sp ? 1 : 0;
    for (int k = 0; k < 6; ++k) a.init_sp[k] = init_sp ? T(init_sp[k]) : T(0);
    a.seed = h->c.seed; a.env_id0 = h->c.env_id0;
    rov6_reset_kernel<T><<<grid_for(n, 128), 128, 0, s>>>(a);
    return check_launch("rov6_reset");
}

extern "C" MVRL_API int mvrl_rov6_reset(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const uint8_t* mask,
                               const double* initial_setpoint_host, mvrl_stream_t stream) {
    if (!h || !b) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_reset: null argument");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_reset: need 0 <= n <= ld");
    if (!b->state || !b->obs || !b->istep || !b->setpoint || !b->path)
        return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_reset: state/obs/istep/setpoint/path are required");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    cudaStream_t s = (cudaStream_t)stream;
    if (h->c.dtype == MVRL_F64) return reset_impl<double>(h, h->pd, n, ld, b, mask, initial_setpoint_host, s);
    return reset_impl<float>(h, h->pf, n, ld, b, mask, initial_setpoint_host, s);
}

template <typename T>
static int pid_impl(const Rov6Dev<T>& P, int64_t n, int64_t ld, const void* pose, const void* t, const void* sp, void* ctrl, void* forces, cudaStream_t s) {
    Rov6PidArgs<T> a;
    a.P = P; a.n = n; a.ld = ld; a.pose = (const T*)pose; a.t = (const T*)t; a.setpoint = (const T*)sp; a.ctrl = (T*)ctrl; a.forces = (T*)forces;
    rov6_pid_kernel<T><<<grid_for(n, 128), 128, 0, s>>>(a);
    return check_launch("rov6_pid");
}

extern "C" MVRL_API int mvrl_rov6_pid(MvrlRov6* h, int64_t n, int64_t ld, const void* pose, const void* t, const void* setpoint,
                             void* ctrl, void* forces, mvrl_stream_t stream) {
    if (!h || !pose || !t || !setpoint || !ctrl || !forces) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_pid: null argument");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_pid: need 0 <= n <= ld");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    if (h->c.dtype == MVRL_F64) return pid_impl<double>(h->pd, n, ld, pose, t, setpoint, ctrl, forces, (cudaStream_t)stream);
    return pid_impl<float>(h->pf, n, ld, pose, t, setpoint, ctrl, forces, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------
// resources.py helpers
// ---------------------------------------------------------------------------
template <typename T>
__global__ void coordinate_transform_kernel(int dof, long n, long ld, const T* phi, const T* theta, const T* psi, T* out) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (dof == 3) {  // resources.py:108-113
        T s, c;
        Real<T>::sincos(psi[i], &s, &c);
        const T J[9] = {c, -s, T(0), s, c, T(0), T(0), T(0), T(1)};
#pragma unroll
        for (int k = 0; k < 9; ++k) out[k * ld + i] = J[k];
        return;
    }
    // resources.py:115-141: J = blkdiag(J1, J2), obtained column by column from kinematics6
    const Trig6<T> g = trig6<T, false>(phi[i], theta[i], psi[i]);
#pragma unroll
    for (int c = 0; c < 6; ++c) {
        T nu[6] = {T(0), T(0), T(0), T(0), T(0), T(0)};
        nu[c] = T(1);
        T ed[6];
        kinematics6<T, false>(g, nu, ed);
#pragma unroll
        for (int r = 0; r < 6; ++r) out[(r * 6 + c) * ld + i] = ed[r];
    }
}

extern "C" MVRL_API int mvrl_coordinate_transform(int dtype, int dof, int64_t n, int64_t ld, const void* phi, const void* theta,
                                         const void* psi, void* out, mvrl_stream_t stream) {
    if ((dof != 3 && dof != 6) || !psi || !out || (dof == 6 && (!phi || !theta))) return mvrl_fail(MVRL_EINVAL, "mvrl_coordinate_transform: bad argument");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_coordinate_transform: need 0 <= n <= ld");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, psi, "mvrl_coordinate_transform");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) coordinate_transform_kernel<double><<<grid_for(n, 128), 128, 0, s>>>(dof, n, ld, (const double*)phi, (const double*)theta, (const double*)psi, (double*)out);
    else if (dtype == MVRL_F32) coordinate_transform_kernel<float><<<grid_for(n, 128), 128, 0, s>>>(dof, n, ld, (const float*)phi, (const float*)theta, (const float*)psi, (float*)out);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return check_launch("coordinate_transform");
}

template <typename T>
__global__ void angle_error_kernel(long n, const T* a, const T* b, T* out) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = angle_error(a[i], b[i]);
}

extern "C" MVRL_API int mvrl_angle_error(int dtype, int64_t n, const void* psi_d, const void* psi, void* out, mvrl_stream_t stream) {
    if (!psi_d || !psi || !out || n < 0) return mvrl_fail(MVRL_EINVAL, "mvrl_angle_error: bad argument");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, psi, "mvrl_angle_error");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) angle_error_kernel<double><<<grid_for(n, 128), 128, 0, s>>>(n, (const double*)psi_d, (const double*)psi, (double*)out);
    else if (dtype == MVRL_F32) angle_error_kernel<float><<<grid_for(n, 128), 128, 0, s>>>(n, (const float*)psi_d, (const float*)psi, (float*)out);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return check_launch("angle_error");
}

template <typename T>
__global__ void body_axes_kernel(long n, long ld, const T* ang, T* out) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Trig6<T> g = trig6<T, false>(ang[i], ang[ld + i], ang[2 * ld + i]);
    // rows of R^T for R = Rx(phi) Ry(theta) Rz(psi), 6DoF.py:242
    const T ax[9] = {g.cth * g.cps, g.cph * g.sps + g.sph * g.sth * g.cps, g.sph * g.sps - g.cph * g.sth * g.cps,
                     -g.cth * g.sps, g.cph * g.cps - g.sph * g.sth * g.sps, g.sph * g.cps + g.cph * g.sth * g.sps,
                     g.sth, -g.sph * g.cth, g.cph * g.cth};
#pragma unroll
    for (int k = 0; k < 9; ++k) out[k * ld + i] = ax[k];
}

extern "C" MVRL_API int mvrl_body_axes(int dtype, int64_t n, int64_t ld, const void* angles, void* out, mvrl_stream_t stream) {
    if (!angles || !out || n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_body_axes: bad argument");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, angles, "mvrl_body_axes");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) body_axes_kernel<double><<<grid_for(n, 128), 128, 0, s>>>(n, ld, (const double*)angles, (double*)out);
    else if (dtype == MVRL_F32) body_axes_kernel<float><<<grid_for(n, 128), 128, 0, s>>>(n, ld, (const float*)angles, (float*)out);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return check_launch("body_axes");
}

// ---------------------------------------------------------------------------
// K6: FP-pipe peak calibration (roofline denominator).  Every thread runs
// CHAINS independent dependent-FMA chains; 2 flop per FMA.  This entry point
// is a measurement utility: it allocates a scratch buffer and synchronises.
// ---------------------------------------------------------------------------
template <typename T, int CHAINS>
__global__ void __launch_bounds__(256) fma_peak_kernel(T* out, int iters, T a, T b) {
    T x[CHAINS];
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) x[j] = T(threadIdx.x + j) * T(1e-3);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int j = 0; j < CHAINS; ++j) x[j] = fmaf_t(x[j], a, b);   // explicit: this unit is built with -fmad=false
        }
    }
    T s = T(0);
#pragma unroll
    for (int j = 0; j < CHAINS; ++j) s += x[j];
    out[(long)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" MVRL_API int mvrl_measure_fma_peak(int dtype, int device, int iters, double* tflops_out, double* ms_out) {
    if (!tflops_out || iters < 1) return mvrl_fail(MVRL_EINVAL, "mvrl_measure_fma_peak: bad argument");
    MVRL_ON_DEVICE(device);
    cudaDeviceProp prop;
    MVRL_CUDA(cudaGetDeviceProperties(&prop, device));
    constexpr int CH = 8;
    const int blocks = prop.multiProcessorCount * 8, threads = 256;
    void* buf = nullptr;
    MVRL_CUDA(cudaMalloc(&buf, (size_t)blocks * threads * 8));
    cudaEvent_t e0, e1;
    MVRL_CUDA(cudaEventCreate(&e0));
    MVRL_CUDA(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 6; ++rep) {  // first reps warm the clocks up; keep the best
        MVRL_CUDA(cudaEventRecord(e0, 0));
        if (dtype == MVRL_F64) fma_peak_kernel<double, CH><<<blocks, threads>>>((double*)buf, iters, 0.999999, 1e-7);
        else fma_peak_kernel<float, CH><<<blocks, threads>>>((float*)buf, iters, 0.999999f, 1e-7f);
        MVRL_CUDA(cudaEventRecord(e1, 0));
        MVRL_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        MVRL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (rep >= 2 && ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    const double flops = 2.0 * CH * 8.0 * (double)iters * (double)blocks * threads;
    *tflops_out = flops / (best * 1e-3) / 1e12;
    if (ms_out) *ms_out = best;
    return check_launch("fma_peak");
}

// ---------------------------------------------------------------------------
// small pieces of the BlueROV2Heavy6DoF surface used by the single-vehicle API
// ---------------------------------------------------------------------------
// thrusterModel(rpm), 6DoF.py:233-236 (no saturation / deadband: those are applied by forceModel)
template <typename T>
__global__ void rov6_thruster_kernel(T thrust_k, long n, const T* rpm, T* F) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) F[i] = thrust_k * rpm[i] * tabs(rpm[i]);
}

extern "C" MVRL_API int mvrl_rov6_thruster_model(MvrlRov6* h, int64_t n, const void* rpm, void* F, mvrl_stream_t stream) {
    if (!h || !rpm || !F || n < 0) return mvrl_fail(MVRL_EINVAL, "mvrl_rov6_thruster_model: bad argument");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    cudaStream_t s = (cudaStream_t)stream;
    if (h->c.dtype == MVRL_F64) rov6_thruster_kernel<double><<<grid_for(n, 128), 128, 0, s>>>(h->pd.thrust_k, n, (const double*)rpm, (double*)F);
    else rov6_thruster_kernel<float><<<grid_for(n, 128), 128, 0, s>>>(h->pf.thrust_k, n, (const float*)rpm, (float*)F);
    return check_launch("rov6_thruster_model");
}

// globalToVehicle (to_vehicle = 1, 6DoF.py:244-248) / vehicleToGlobal (0, 6DoF.py:250-251)
template <typename T>
__global__ void frame_rotate_kernel(long n, long ld, const T* axes, const T* v, T* out, int to_vehicle) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T ax[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) ax[k] = axes[k * ld + i];
    const T a = v[i], b = v[ld + i], c = v[2 * ld + i];
    if (to_vehicle) {
        out[i] = a * ax[0] + b * ax[1] + c * ax[2];
        out[ld + i] = a * ax[3] + b * ax[4] + c * ax[5];
        out[2 * ld + i] = a * ax[6] + b * ax[7] + c * ax[8];
    } else {
        out[i] = a * ax[0] + b * ax[3] + c * ax[6];
        out[ld + i] = a * ax[1] + b * ax[4] + c * ax[7];
        out[2 * ld + i] = a * ax[2] + b * ax[5] + c * ax[8];
    }
}

extern "C" MVRL_API int mvrl_frame_rotate(int dtype, int64_t n, int64_t ld, const void* axes, const void* v, void* out, int to_vehicle,
                                          mvrl_stream_t stream) {
    if (!axes || !v || !out || n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_frame_rotate: bad argument");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, v, "mvrl_frame_rotate");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) frame_rotate_kernel<double><<<grid_for(n, 128), 128, 0, s>>>(n, ld, (const double*)axes, (const double*)v, (double*)out, to_vehicle);
    else if (dtype == MVRL_F32) frame_rotate_kernel<float><<<grid_for(n, 128), 128, 0, s>>>(n, ld, (const float*)axes, (const float*)v, (float*)out, to_vehicle);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return check_launch("frame_rotate");
}
