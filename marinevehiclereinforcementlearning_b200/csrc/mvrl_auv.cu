// C ABI of the legacy path (K4): AuvEnv step/reset and ReconstructedFlow scale/interp.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "mvrl_host.h"
#include "auv_kernels.cuh"

using namespace mvrl;

struct MvrlAuv {
    MvrlAuvParams p;
    MvrlAuvConfig c;
    const void* field;
    int nt, ny, nx, nc;
    double dx, dy, dtf;
    bool stage_smem;   // MVRL_AUV_NO_STAGE=1 in the environment selects the direct L2 gather instead
};

extern "C" MVRL_API int mvrl_auv_default_params(MvrlAuvParams* p) {
    if (!p) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_default_params: null output");
    // verySimpleAuv.py:110-132
    p->m = 11.4; p->Izz = 0.16;
    p->Xuu = -18.18 * 2.21; p->Yvv = -21.66 * 4.87; p->Nrr = -1.55;
    p->Xu = -4.03 * 2.21; p->Yv = -6.22 * 4.87; p->Nr = -0.07;
    p->maxForce = 150.; p->maxMoment = 20.;
    p->xMin = -1.; p->xMax = 1.; p->yMin = -1.; p->yMax = 1.;
    p->noiseMagCoeffs = 0.; p->noiseMagActuation = 0.;
    p->variant = MVRL_AUV_PLAIN; p->n_waypoints = 0; p->wp_threshold = 0.;
    memset(p->waypoints, 0, sizeof(p->waypoints));
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_auv_create(MvrlAuv** out, const MvrlAuvParams* params, const MvrlAuvConfig* cfg) {
    if (!out || !params || !cfg) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_create: null argument");
    if (cfg->dtype != MVRL_F32 && cfg->dtype != MVRL_F64) return mvrl_fail(MVRL_EINVAL, "dtype must be MVRL_F32 or MVRL_F64");
    if (!(cfg->dt > 0)) return mvrl_fail(MVRL_EINVAL, "dt must be > 0");
    if (params->variant == MVRL_AUV_CYL && (params->n_waypoints < 1 || params->n_waypoints > 32))
        return mvrl_fail(MVRL_EINVAL, "AuvEnvCyl needs 1..32 way-points");
    if (params->variant != MVRL_AUV_CYL && params->variant != MVRL_AUV_PLAIN) return mvrl_fail(MVRL_EINVAL, "bad variant");
    { const int rc = mvrl_require_device(cfg->device); if (rc != MVRL_OK) return rc; }
    MvrlAuv* h = new (std::nothrow) MvrlAuv();
    if (!h) return mvrl_fail(MVRL_EINVAL, "out of host memory");
    h->p = *params; h->c = *cfg; h->field = nullptr;
    { const char* e = getenv("MVRL_AUV_NO_STAGE"); h->stage_smem = !(e && e[0] == '1'); }
    *out = h;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_auv_destroy(MvrlAuv* h) { delete h; return MVRL_OK; }

extern "C" MVRL_API int mvrl_auv_set_apply_noise(MvrlAuv* h, int apply_noise) {
    if (!h) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_set_apply_noise: null handle");
    h->c.apply_noise = apply_noise ? 1 : 0;
    return MVRL_OK;
}

extern "C" MVRL_API int mvrl_auv_set_flow(MvrlAuv* h, const void* field, int nt, int ny, int nx, int nc, double dx, double dy, double dt) {
    if (!h || !field) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_set_flow: null argument");
    if (nt < 2 || ny < 2 || nx < 2 || (nc != 2 && nc != 3)) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_set_flow: need nt, ny, nx >= 2 and nc in {2, 3}");
    if (!(dx > 0) || !(dy > 0) || !(dt > 0)) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_set_flow: spacings must be > 0");
    h->field = field; h->nt = nt; h->ny = ny; h->nx = nx; h->nc = nc; h->dx = dx; h->dy = dy; h->dtf = dt;
    return MVRL_OK;
}

template <typename T> static FlowDev<T> flow_dev(const void* field, int nt, int ny, int nx, int nc, double dx, double dy, double dt) {
    FlowDev<T> f;
    f.field = (const T*)field; f.nt = nt; f.ny = ny; f.nx = nx; f.nc = nc; f.dx = T(dx); f.dy = T(dy); f.dt = T(dt);
    f.inv_dx = T(1. / dx); f.inv_dy = T(1. / dy); f.inv_dt = T(1. / dt);
    return f;
}

template <typename T> static AuvDev<T> auv_dev(const MvrlAuv* h) {
    const MvrlAuvParams& p = h->p;
    AuvDev<T> d;
    d.m = T(p.m); d.Izz = T(p.Izz); d.Xuu = T(p.Xuu); d.Yvv = T(p.Yvv); d.Nrr = T(p.Nrr); d.Xu = T(p.Xu); d.Yv = T(p.Yv); d.Nr = T(p.Nr);
    d.maxForce = T(p.maxForce); d.maxMoment = T(p.maxMoment);
    d.xmin = T(p.xMin); d.xmax = T(p.xMax); d.ymin = T(p.yMin); d.ymax = T(p.yMax);
    d.noise_coeffs = T(p.noiseMagCoeffs); d.noise_act = T(p.noiseMagActuation);
    d.t_quarter = T((double)(h->nt / 4) * h->dtf);  // flow.time[nt // 4], verySimpleAuv.py:245
    d.cyl = p.variant == MVRL_AUV_CYL ? 1 : 0; d.n_wp = p.n_waypoints; d.wp_thr = T(p.wp_threshold);
    for (int k = 0; k < 32; ++k) for (int j = 0; j < 3; ++j) d.wp[k][j] = T(k < p.n_waypoints ? p.waypoints[k * 3 + j] : 0.);
    return d;
}

template <typename T> static int auv_step_impl(const MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, cudaStream_t s) {
    AuvStepArgs<T> a;
    a.P = auv_dev<T>(h);
    a.flow = flow_dev<T>(h->field, h->nt, h->ny, h->nx, h->nc, h->dx, h->dy, h->dtf);
    a.n = n; a.ld = ld;
    a.state = (T*)b->state; a.action = (const T*)b->action; a.obs = (T*)b->obs; a.reward = (T*)b->reward; a.done = b->done; a.istep = b->istep;
    a.mults = (T*)b->mults; a.target = (T*)b->target; a.err_o = (T*)b->err_o; a.recent = (T*)b->recent; a.ep_return = (T*)b->ep_return;
    a.iwp = b->iwp;
    a.episode = b->episode; a.term_obs = (T*)b->terminal_obs; a.aux = (T*)b->aux; a.stats = b->ep_stats;
    a.dt = T(h->c.dt); a.max_steps = h->c.max_steps; a.seed = h->c.seed; a.env_id0 = h->c.env_id0;
    a.auto_reset = h->c.auto_reset; a.stop_on_bounds = h->c.stop_on_bounds; a.apply_noise = h->c.apply_noise;
    if constexpr (sizeof(T) == 4) {
        // staged gather needs the interleaved (u, v) field, 8-byte aligned
        if (h->nc == 2 && (((uintptr_t)h->field) & 7u) == 0 && h->stage_smem) {
            if (a.P.cyl) auv_step_kernel<T, true, true><<<mvrl_grid_for(n, AUV_BLOCK), AUV_BLOCK, 0, s>>>(a);
            else auv_step_kernel<T, true, false><<<mvrl_grid_for(n, AUV_BLOCK), AUV_BLOCK, 0, s>>>(a);
            return mvrl_check_launch("auv_step");
        }
    }
    if (a.P.cyl) auv_step_kernel<T, false, true><<<mvrl_grid_for(n, AUV_BLOCK), AUV_BLOCK, 0, s>>>(a);
    else auv_step_kernel<T, false, false><<<mvrl_grid_for(n, AUV_BLOCK), AUV_BLOCK, 0, s>>>(a);
    return mvrl_check_launch("auv_step");
}

extern "C" MVRL_API int mvrl_auv_step(MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, mvrl_stream_t stream) {
    if (!h || !b) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: null argument");
    if (!h->field) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: call mvrl_auv_set_flow first");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: need 0 <= n <= ld");
    if (!b->state || !b->action || !b->obs || !b->reward || !b->done || !b->istep || !b->mults || !b->target || !b->err_o || !b->recent || !b->ep_return)
        return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: missing required buffer");
    if (h->c.auto_reset && !b->episode) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: episode is required with auto_reset");
    if (h->p.variant == MVRL_AUV_CYL && !b->iwp) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_step: iwp is required for the AuvEnvCyl variant");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    if (h->c.dtype == MVRL_F64) return auv_step_impl<double>(h, n, ld, b, (cudaStream_t)stream);
    return auv_step_impl<float>(h, n, ld, b, (cudaStream_t)stream);
}

template <typename T> static int auv_reset_impl(const MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, const uint8_t* mask, const void* init, cudaStream_t s) {
    AuvResetArgs<T> a;
    a.P = auv_dev<T>(h);
    a.n = n; a.ld = ld;
    a.state = (T*)b->state; a.obs = (T*)b->obs; a.istep = b->istep; a.mults = (T*)b->mults; a.target = (T*)b->target; a.err_o = (T*)b->err_o;
    a.recent = (T*)b->recent; a.ep_return = (T*)b->ep_return; a.iwp = b->iwp; a.episode = b->episode; a.mask = mask; a.init = (const T*)init;
    a.seed = h->c.seed; a.env_id0 = h->c.env_id0; a.apply_noise = h->c.apply_noise;
    auv_reset_kernel<T><<<mvrl_grid_for(n, 128), 128, 0, s>>>(a);
    return mvrl_check_launch("auv_reset");
}

extern "C" MVRL_API int mvrl_auv_reset(MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, const uint8_t* mask, const void* init, mvrl_stream_t stream) {
    if (!h || !b) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_reset: null argument");
    if (!h->field) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_reset: call mvrl_auv_set_flow first (the time offset is drawn from the field's time range)");
    if (n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_reset: need 0 <= n <= ld");
    if (!b->state || !b->obs || !b->istep || !b->mults || !b->target || !b->err_o || !b->recent || !b->ep_return)
        return mvrl_fail(MVRL_EINVAL, "mvrl_auv_reset: missing required buffer");
    if (h->p.variant == MVRL_AUV_CYL && !b->iwp) return mvrl_fail(MVRL_EINVAL, "mvrl_auv_reset: iwp is required for the AuvEnvCyl variant");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE(h->c.device);
    if (h->c.dtype == MVRL_F64) return auv_reset_impl<double>(h, n, ld, b, mask, init, (cudaStream_t)stream);
    return auv_reset_impl<float>(h, n, ld, b, mask, init, (cudaStream_t)stream);
}

extern "C" MVRL_API int mvrl_flow_interp(int dtype, const void* field, int nt, int ny, int nx, int nc, double dx, double dy, double dt,
                                         int64_t n, int64_t ld, const void* t, const void* xy, void* out, mvrl_stream_t stream) {
    if (!field || !t || !xy || !out || n < 0 || ld < n) return mvrl_fail(MVRL_EINVAL, "mvrl_flow_interp: bad argument");
    if (nt < 2 || ny < 2 || nx < 2 || (nc != 2 && nc != 3)) return mvrl_fail(MVRL_EINVAL, "mvrl_flow_interp: need nt, ny, nx >= 2 and nc in {2, 3}");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, field, "mvrl_flow_interp");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) flow_interp_kernel<double><<<mvrl_grid_for(n, 128), 128, 0, s>>>(flow_dev<double>(field, nt, ny, nx, nc, dx, dy, dt), n, ld, (const double*)t, (const double*)xy, (double*)out);
    else if (dtype == MVRL_F32) flow_interp_kernel<float><<<mvrl_grid_for(n, 128), 128, 0, s>>>(flow_dev<float>(field, nt, ny, nx, nc, dx, dy, dt), n, ld, (const float*)t, (const float*)xy, (float*)out);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return mvrl_check_launch("flow_interp");
}

extern "C" MVRL_API int mvrl_flow_scale(int dtype, int64_t cells, const void* base, void* out, int nc_out, double velocityScale,
                                        double turbScale, mvrl_stream_t stream) {
    if (!base || !out || cells < 0 || (nc_out != 2 && nc_out != 3)) return mvrl_fail(MVRL_EINVAL, "mvrl_flow_scale: bad argument");
    if (cells == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(out, base, "mvrl_flow_scale");
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) flow_scale_kernel<double><<<mvrl_grid_for(cells, 256), 256, 0, s>>>(cells, (const double*)base, (double*)out, nc_out, velocityScale, turbScale);
    else if (dtype == MVRL_F32) flow_scale_kernel<float><<<mvrl_grid_for(cells, 256), 256, 0, s>>>(cells, (const float*)base, (float*)out, nc_out, (float)velocityScale, (float)turbScale);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return mvrl_check_launch("flow_scale");
}

extern "C" MVRL_API int mvrl_flow_reconstruct(int dtype, int64_t plane, int n_modes, int nt, const double* modes, int modes_complex,
                                              const double* coeffs, int coeffs_complex, const double* mean, void* out, mvrl_stream_t stream) {
    if (!modes || !coeffs || !mean || !out) return mvrl_fail(MVRL_EINVAL, "mvrl_flow_reconstruct: null argument");
    if (plane < 1 || n_modes < 1 || nt < 1) return mvrl_fail(MVRL_EINVAL, "mvrl_flow_reconstruct: plane, n_modes and nt must be >= 1");
    if (dtype != MVRL_F32 && dtype != MVRL_F64) return mvrl_fail(MVRL_EINVAL, "bad dtype");
    MVRL_ON_DEVICE_OF(out, modes, "mvrl_flow_reconstruct");
    if (mvrl_device_of(coeffs) != mvrl_dev_out_ || mvrl_device_of(mean) != mvrl_dev_out_)
        return mvrl_fail(MVRL_EINVAL, "mvrl_flow_reconstruct: coeffs / mean are not on the output's device");
    const dim3 grid((unsigned)((plane + 127) / 128), (unsigned)((nt + 63) / 64));
    cudaStream_t s = (cudaStream_t)stream;
    if (dtype == MVRL_F64) flow_reconstruct_kernel<double><<<grid, 256, 0, s>>>(plane, n_modes, nt, modes, modes_complex, coeffs, coeffs_complex, mean, (double*)out);
    else flow_reconstruct_kernel<float><<<grid, 256, 0, s>>>(plane, n_modes, nt, modes, modes_complex, coeffs, coeffs_complex, mean, (float*)out);
    return mvrl_check_launch("flow_reconstruct");
}

extern "C" MVRL_API int mvrl_replay_add_symmetric(int dtype, int64_t n, int64_t ld, const void* obs, const void* next_obs, const void* act,
                                                  const void* reward, const uint8_t* done, const uint8_t* timeout, void* buf_obs, void* buf_next_obs,
                                                  void* buf_act, void* buf_reward, uint8_t* buf_done, uint8_t* buf_timeout, int64_t buffer_size,
                                                  int64_t pos, int n_transforms, mvrl_stream_t stream) {
    if (!obs || !next_obs || !act || !reward || !done || !buf_obs || !buf_next_obs || !buf_act || !buf_reward || !buf_done)
        return mvrl_fail(MVRL_EINVAL, "mvrl_replay_add_symmetric: null argument");
    if (n < 0 || ld < n || buffer_size < 1 || pos < 0 || pos >= buffer_size || n_transforms < 1 || n_transforms > 5 || n_transforms > buffer_size)
        return mvrl_fail(MVRL_EINVAL, "mvrl_replay_add_symmetric: bad size argument");
    if (n == 0) return MVRL_OK;
    MVRL_ON_DEVICE_OF(buf_obs, obs, "mvrl_replay_add_symmetric");
    cudaStream_t s = (cudaStream_t)stream;
    const unsigned g = mvrl_grid_for(n * n_transforms, 256);
    if (dtype == MVRL_F64)
        replay_add_symmetric_kernel<double><<<g, 256, 0, s>>>(n, ld, (const double*)obs, (const double*)next_obs, (const double*)act, (const double*)reward,
                                                              done, timeout, (double*)buf_obs, (double*)buf_next_obs, (double*)buf_act, (double*)buf_reward,
                                                              buf_done, buf_timeout, buffer_size, pos, n_transforms);
    else if (dtype == MVRL_F32)
        replay_add_symmetric_kernel<float><<<g, 256, 0, s>>>(n, ld, (const float*)obs, (const float*)next_obs, (const float*)act, (const float*)reward,
                                                             done, timeout, (float*)buf_obs, (float*)buf_next_obs, (float*)buf_act, (float*)buf_reward,
                                                             buf_done, buf_timeout, buffer_size, pos, n_transforms);
    else return mvrl_fail(MVRL_EINVAL, "bad dtype");
    return mvrl_check_launch("replay_add_symmetric");
}
