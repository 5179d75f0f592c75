/*
 * mvrl.h - C ABI of libmvrl.so: B200-native batched BlueROV2 Heavy simulator.
 *
 * The reference (UnnamedMoose/MarineVehicleReinforcementLearning) is pure
 * Python and has no FFI layer; its "operator interface" for this path is the
 * Python class surface.  Each entry point below replaces the per-environment
 * numpy code of one reference function, batched over N environments:
 *
 *   mvrl_rov6_derivs      BlueROV2Heavy6DoF.derivs / forceModel / allocateThrust
 *                         dynamicsModel_BlueROV2_Heavy_6DoF.py:220-236, 253-442
 *   mvrl_rov6_step        BlueROV2Heavy6DoFEnv.step + dataToState
 *                         dynamicsModel_BlueROV2_Heavy_6DoF.py:467-483, 531-594
 *   mvrl_rov6_reset       BlueROV2Heavy6DoFEnv.reset
 *                         dynamicsModel_BlueROV2_Heavy_6DoF.py:485-529
 *   mvrl_rov6_pid         BlueROV2Heavy6DoF_PID_controller.computeControlForces
 *                         dynamicsModel_BlueROV2_Heavy_6DoF.py:43-73
 *   mvrl_coordinate_transform / mvrl_angle_error / mvrl_body_axes
 *                         resources.py:98-143 / resources.py:75-95 /
 *                         dynamicsModel_BlueROV2_Heavy_6DoF.py:238-251
 *   mvrl_rov3_*           dynamicsModel_BlueROV2_Heavy_3DoF.py:114-296, 397-514
 *   mvrl_auv_*            tag_00_Dec2023_simpleControlTurbulence/verySimpleAuv.py:147-410
 *                         and flowGenerator.py:53-136
 *
 * Conventions
 *   - every function returns 0 on success and a negative MVRL_E* code on
 *     failure; mvrl_last_error() returns a thread-local message.  No C++
 *     exception crosses this boundary.
 *   - all array pointers are DEVICE pointers on the handle's device unless the
 *     name says "host".  Arrays are structure-of-arrays: field k of
 *     environment i lives at base[k * ld + i] (ld >= n, the leading dimension).
 *     Element type is float (dtype 0) or double (dtype 1) as fixed at create.
 *   - the library allocates nothing per call, never synchronises, and launches
 *     on the caller's stream (CUDA-graph capturable).
 *   - a handle is not thread-safe; use one per GPU / process.
 */
#ifndef MVRL_H_
#define MVRL_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MVRL_VERSION 100

#define MVRL_OK 0
#define MVRL_EINVAL (-1)   /* bad argument */
#define MVRL_ECUDA (-2)    /* CUDA runtime error (message has the detail) */
#define MVRL_ENODEV (-3)   /* no usable CUDA device */

#define MVRL_F32 0
#define MVRL_F64 1

/* action semantics of the 6DoF step */
#define MVRL_ACT_RPM 0       /* action = 8 thruster rpm (synthetic random-thruster workload) */
#define MVRL_ACT_FORCE 1     /* action = 6 earth-frame generalised forces (stateless controller seam) */
#define MVRL_ACT_SETPOINT 2  /* action in [-1,1]^6 -> PID set-point: the reference's Gym semantics */

typedef void* mvrl_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define MVRL_API __attribute__((visibility("default")))
#else
#define MVRL_API
#endif

/* ---------------------------------------------------------------- 6DoF -- */

/* Physical + derived constants of BlueROV2Heavy6DoF
 * (dynamicsModel_BlueROV2_Heavy_6DoF.py:83-218).  Names follow the reference.
 * Derived matrices are supplied by the host so that they are bit-identical to
 * what numpy gives the reference (pinv / inv); mvrl_rov6_default_params fills
 * everything natively for non-Python callers. */
typedef struct MvrlRov6Params {
    double rho_f, m, Length;
    double CG[3], CB[3];
    double I[9];                                  /* row-major 3x3 */
    double Xudot, Yvdot, Zwdot, Kpdot, Mqdot, Nrdot; /* used by Ca (6DoF.py:334-341) */
    /* linear damping, 6DoF.py:345-352 */
    double Xu, Yv, Yp, Yr, Zw, Zq, Kv, Kp, Kr, Mw, Mq, Nv, Np, Nr;
    /* quadratic damping, 6DoF.py:354-368 */
    double Xuu, Yvv, Ypp, Yrr, Zww, Zqq, Kvv, Kpp, Krr, Mww, Mqq, Nvv, Npp, Nrr;
    double W, B;                                  /* weight m*9.81 and buoyancy dispVol*rho_f*9.81 */
    double thrust_coef;                           /* rho_f * D_thruster^4 * Kt_thruster */
    double rpm_max, rpm_deadband;                 /* 3500, 300 (6DoF.py:271-275) */
    double M[36];                                 /* Mrb + Ma, row-major (6DoF.py:286-299) */
    double Minv[36];                              /* inverse of M */
    double A[48];                                 /* 6x8 allocation matrix, row-major (resources.py:19-35) */
    double Ainv[48];                              /* 8x6 pseudo-inverse, row-major */
    /* PID controller, 6DoF.py:46-54 */
    double pid_Kp[6], pid_Ki[6], pid_Kd[6], pid_windup[6], pid_max[6];
    int disable_thrusters;                        /* BlueROV2Heavy6DoF(disableThrusters=...) */
} MvrlRov6Params;

typedef struct MvrlRov6Config {
    int dtype;         /* MVRL_F32 / MVRL_F64 */
    int action_mode;   /* MVRL_ACT_* */
    int n_sub;         /* RK4 sub-steps per env step (>= 1) */
    int max_steps;     /* done when iStep >= max_steps (6DoF.py:569-571) */
    double dt;         /* env step, 0.2 in the reference */
    uint64_t seed;     /* Philox key for the random reset branch */
    uint64_t env_id0;  /* global id of environment 0 of this shard (results independent of sharding) */
    int auto_reset;    /* 1: SB3-VecEnv style reset inside the step kernel; 0: reference behaviour */
    int fixed_sp;      /* 1: reset(initialSetpoint=...) mode, actions ignored (6DoF.py:536-541) */
    int device;        /* CUDA device ordinal */
    int fast_math;     /* fp32 only: 1 = MUFU sin/cos + approximate reciprocal */
} MvrlRov6Config;

/* Device buffers of one batch of 6DoF environments.  T = element type.
 * Nullable members may be NULL.  Every row must be allocated to its full leading dimension ld (ld >= n):
 * the fp32 kernels that carry two environments per thread access rows in 8-byte units, so the padding element
 * after an odd n is read (never written).  That path needs ld even and 8-byte aligned rows (2-byte for done);
 * other layouts silently take the one-environment-per-thread kernels. */
typedef struct MvrlRov6Buffers {
    void* state;        /* T [12][ld] x y z phi theta psi u v w p q r       in/out */
    void* action;       /* T [8|6][ld] per action_mode                       in     */
    void* obs;          /* T [9][ld]  6DoF.py:467-483                        out    */
    void* reward;       /* T [ld]     (identically 0, 6DoF.py:575)           out    */
    uint8_t* done;      /* [ld]                                              out    */
    int32_t* istep;     /* [ld]       iStep                                  in/out */
    void* setpoint;     /* T [6][ld]  controller.setPoint                    in/out */
    void* path;         /* T [6][ld]  path[0,:], path[1,:]                   in (out on reset) */
    void* ctrl;         /* T [13][ld] eOld(6) eInt(6) tOld; eOld[0]=NaN <=> eOld is None;
                           required for MVRL_ACT_SETPOINT, else nullable     in/out */
    uint32_t* episode;  /* [ld] episode counter (Philox stream); nullable iff !auto_reset */
    void* terminal_obs; /* T [9][ld] obs before auto-reset, written where done; nullable */
    void* aux;          /* T [14][ld] generalisedControlForces(6), controlVector(8) of the
                           last derivative evaluation (6DoF.py:578-580); nullable */
    double* ep_stats;   /* [8]: episodes, sum length, sum return, min return, max return,
                           non-finite states, 0, 0 - accumulated atomically; nullable */
} MvrlRov6Buffers;

typedef struct MvrlRov6 MvrlRov6;

MVRL_API int mvrl_version(void);
MVRL_API const char* mvrl_last_error(void);
MVRL_API int mvrl_device_count(void);

MVRL_API int mvrl_rov6_default_params(MvrlRov6Params* out);
MVRL_API int mvrl_rov6_create(MvrlRov6** out, const MvrlRov6Params* params, const MvrlRov6Config* cfg);
MVRL_API int mvrl_rov6_destroy(MvrlRov6* h);
/* 1 if the handle runs the kernels specialised for the reference's default
 * sparsity pattern (CG on the z axis, diagonal inertia, no cross damping but
 * Mww, neutral buoyancy, default allocation pattern), 0 for the generic ones;
 * 2 if, in addition, its fp32 constants equal the compiled-in default vehicle
 * (6DoF.py:83-218) bit for bit, so that the fp32 step kernels with literal
 * constants are used (same results, fewer instructions) */
MVRL_API int mvrl_rov6_is_specialised(const MvrlRov6* h);
/* The fp32 device constants a parameter set converts to, flattened (build-time helper of
 * tools/gen_default_consts.py, which writes csrc/rov6_default_consts.h).  Returns the number of floats. */
MVRL_API int mvrl_rov6_dev_constants_f32(const MvrlRov6Params* params, float* out, int capacity);

/* One derivative evaluation per environment (debug / parity entry, K2).
 *   state  T [12][ld]; dstate T [12][ld]
 *   act    per action_mode: rpm T [8][ld] | force T [6][ld] | (SETPOINT) unused
 *   t      T [ld], setpoint T [6][ld], ctrl T [13][ld]: SETPOINT mode only (ctrl is
 *          updated exactly like the reference mutates its controller, 6DoF.py:62-71)
 *   aux    nullable T [50][ld]: RHS(6) gcf(6) rpm(8) then the five retComp columns
 *          -Crb v, -Ca v, -D v, G, H (6 each), 6DoF.py:401-402 */
MVRL_API int mvrl_rov6_derivs(MvrlRov6* h, int64_t n, int64_t ld, const void* state, const void* act,
                     const void* t, const void* setpoint, void* ctrl, void* dstate, void* aux,
                     mvrl_stream_t stream);

/* One env step for n environments (K1). */
MVRL_API int mvrl_rov6_step(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, mvrl_stream_t stream);

/* Same for the environments [first, first + n) of the buffers only (all arrays keep leading dimension ld;
 * the Philox stream of environment first + i is that of global id env_id0 + first + i).  Lets host code
 * build its own copy/compute pipelines over pieces of one batch. */
MVRL_API int mvrl_rov6_step_range(MvrlRov6* h, int64_t first, int64_t n, int64_t ld, const MvrlRov6Buffers* b, mvrl_stream_t stream);

/* One env step with HOST buffers - the call a host-side VecEnv user makes (BlueROV2Heavy6DoFEnv.step for n
 * vehicles, 6DoF.py:531-594): actions_host T [n][A] (row = environment) in; obs_host T [n][9], reward_host
 * T [n] (nullable), done_host [n] (nullable) out.  Pinned host memory is needed for the copies to overlap.
 * The batch is cut into `chunks` equal pieces (0: the default - 8, fewer for batches under 512 Ki environments); upload, transpose to SoA, fused step, transpose
 * back and download of different pieces overlap on streams owned by the handle (PCIe is full duplex).  The
 * observations travel by copy engine; the done flags (1 B per environment) are stored straight into done_host by
 * the transpose kernel when that array is pinned, so that the download engine has one copy per piece to do (a
 * pageable array is copied like the observations).  The reward of this env is identically 0 (6DoF.py:575) and does
 * NOT travel: reward_host is zero-filled on the host side - on every call with chunks < 0, and when the pipeline for
 * this set of pointers is captured otherwise; a caller that scribbles on it between calls must clear it again.
 * The whole pipeline is captured into a CUDA graph once per distinct set of pointers (4 cached) and
 * replayed with one launch; chunks < 0 queues |chunks| pieces directly on the streams instead.
 * Device staging buffers are allocated on first use.  Starts after the work queued on `stream` and returns
 * when the host buffers are complete (synchronises `stream`).  b->action is used as the SoA scratch. */
MVRL_API int mvrl_rov6_step_host(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const void* actions_host,
                                 void* obs_host, void* reward_host, uint8_t* done_host, int chunks, mvrl_stream_t stream);

/* Number of pieces mvrl_rov6_step_host cuts a batch of n environments into for a given `chunks` argument
 * (each piece costs 3 kernel launches, 1 upload and 1-3 downloads). */
MVRL_API int mvrl_host_chunk_count(int64_t n, int chunks);

/* reset(): mask nullable (= all).  initial_setpoint: 6 host doubles or NULL for
 * the random branch (path and target orientation drawn from Philox). */
MVRL_API int mvrl_rov6_reset(MvrlRov6* h, int64_t n, int64_t ld, const MvrlRov6Buffers* b, const uint8_t* mask,
                    const double* initial_setpoint_host, mvrl_stream_t stream);

/* Stand-alone PID evaluation: pose T [6][ld], t T [ld], setpoint T [6][ld],
 * ctrl T [13][ld] in/out, forces T [6][ld] out. */
MVRL_API int mvrl_rov6_pid(MvrlRov6* h, int64_t n, int64_t ld, const void* pose, const void* t, const void* setpoint,
                  void* ctrl, void* forces, mvrl_stream_t stream);

/* BlueROV2Heavy6DoF.thrusterModel(rpm) (6DoF.py:233-236): rpm T [n] -> F T [n]; no saturation/deadband */
MVRL_API int mvrl_rov6_thruster_model(MvrlRov6* h, int64_t n, const void* rpm, void* F, mvrl_stream_t stream);
/* globalToVehicle (to_vehicle = 1) / vehicleToGlobal (0), 6DoF.py:244-251:
 * axes T [9][ld] (iHat jHat kHat from mvrl_body_axes), v T [3][ld] -> out T [3][ld] */
MVRL_API int mvrl_frame_rotate(int dtype, int64_t n, int64_t ld, const void* axes, const void* v, void* out, int to_vehicle,
                               mvrl_stream_t stream);

/* ------------------------------------------------------- resources.py -- */
/* J(phi,theta,psi): out T [dof*dof][ld] row-major entries, dof = 3 or 6 */
MVRL_API int mvrl_coordinate_transform(int dtype, int dof, int64_t n, int64_t ld, const void* phi, const void* theta,
                              const void* psi, void* out, mvrl_stream_t stream);
MVRL_API int mvrl_angle_error(int dtype, int64_t n, const void* psi_d, const void* psi, void* out, mvrl_stream_t stream);
/* iHat jHat kHat: out T [9][ld] */
MVRL_API int mvrl_body_axes(int dtype, int64_t n, int64_t ld, const void* angles /* T [3][ld] */, void* out,
                   mvrl_stream_t stream);

/* ---------------------------------------------------------------- 3DoF -- */

/* Constants of BlueROV2Heavy3DoF (dynamicsModel_BlueROV2_Heavy_3DoF.py:39-112). */
typedef struct MvrlRov3Params {
    double rho_f, m, Length, dispVol;
    double xg, yg, Izz;                       /* CG[0], CG[1], I[2,2] */
    double Xudot, Yvdot, Nrdot;
    double Xu, Yv, Yr, Nv, Nr;                /* 3DoF.py:225-229 */
    double Xuu, Yvv, Yrr, Nvv, Nrr;           /* 3DoF.py:231-239 */
    double D_thruster, thrust_coef;           /* thrust_coef = rho_f D^4 Kt */
    double alphaThruster, l_x, l_y;           /* 3DoF.py:89-91 */
    double rpm_max, rpm_deadband;
    double M[9], Minv[9];                     /* 3DoF.py:198-206 and its inverse */
    double Ainv[12];                          /* 4x3 pseudo-inverse, row-major (3DoF.py:104-112) */
    double pid_Kp[3], pid_Ki[3], pid_Kd[3], pid_windup[3], pid_max[3]; /* 3DoF.py:142-154 */
} MvrlRov3Params;

/* action_mode: MVRL_ACT_RPM (4 thruster rpm FP AP FS AS; stateless) or
 * MVRL_ACT_SETPOINT (the reference's semantics, 3DoF.py:466-472). */
typedef MvrlRov6Config MvrlRov3Config;

typedef struct MvrlRov3Buffers {
    void* state;        /* T [6][ld] x y psi u v r                         in/out */
    void* action;       /* T [4|3][ld]                                     in     */
    void* obs;          /* T [5][ld]  3DoF.py:397-409                      out    */
    void* reward;       /* T [ld]                                          out    */
    uint8_t* done;      /* [ld]                                            out    */
    int32_t* istep;     /* [ld]                                            in/out */
    void* setpoint;     /* T [3][ld]                                       in/out */
    void* path;         /* T [4][ld]  path[0,:], path[1,:]                 in (out on reset) */
    void* ctrl;         /* T [7][ld]  eOld(3) eInt(3) tOld; eOld[0]=NaN <=> None */
    uint32_t* episode;  /* [ld] */
    void* terminal_obs; /* T [5][ld], nullable */
    void* aux;          /* T [7][ld] generalisedControlForces(3), controlVector(4); nullable */
    double* ep_stats;   /* [8], nullable */
} MvrlRov3Buffers;

typedef struct MvrlRov3 MvrlRov3;

MVRL_API int mvrl_rov3_default_params(MvrlRov3Params* out);
MVRL_API int mvrl_rov3_create(MvrlRov3** out, const MvrlRov3Params* params, const MvrlRov3Config* cfg);
MVRL_API int mvrl_rov3_destroy(MvrlRov3* h);
/* derivs: act = rpm T [4][ld] (RPM mode) or t/setpoint/ctrl (SETPOINT mode); aux nullable T [7][ld] */
MVRL_API int mvrl_rov3_derivs(MvrlRov3* h, int64_t n, int64_t ld, const void* state, const void* act, const void* t,
                              const void* setpoint, void* ctrl, void* dstate, void* aux, mvrl_stream_t stream);
MVRL_API int mvrl_rov3_step(MvrlRov3* h, int64_t n, int64_t ld, const MvrlRov3Buffers* b, mvrl_stream_t stream);
MVRL_API int mvrl_rov3_reset(MvrlRov3* h, int64_t n, int64_t ld, const MvrlRov3Buffers* b, const uint8_t* mask,
                             const double* initial_setpoint_host /* 3 or NULL */, mvrl_stream_t stream);
/* BlueROV2Heavy3DoF.thrusterModel(u, v, rpm) -> (Fthruster, Xthruster), 3DoF.py:114-126 */
MVRL_API int mvrl_rov3_thruster_model(MvrlRov3* h, int64_t n, const void* u, const void* rpm, void* F, void* X,
                                      mvrl_stream_t stream);

/* LOSNavigation.predict / lineOfSight (3DoF.py:517-607), the heuristic agent in front of the 3DoF env:
 * obs T [5][ld] (way-points relative to the vehicle, heading error) -> action T [3][ld]; rnav = 0.5 upstream */
MVRL_API int mvrl_los_navigation(int dtype, int64_t n, int64_t ld, const void* obs, void* action, double rnav, mvrl_stream_t stream);

/* -------------------------------------------------------------- legacy -- */

/* AuvEnv constants, tag_00.../verySimpleAuv.py:110-132 */
#define MVRL_AUV_PLAIN 0   /* AuvEnv: target at the origin, V3 observation */
#define MVRL_AUV_CYL 1     /* AuvEnvCyl (verySimpleAuv_cyl.py:22-345): way-point list, V0 observation scaling */
typedef struct MvrlAuvParams {
    double m, Izz, Xuu, Yvv, Nrr, Xu, Yv, Nr, maxForce, maxMoment;
    double xMin, xMax, yMin, yMax;
    double noiseMagCoeffs, noiseMagActuation;
    double wp_threshold;          /* AuvEnvCyl: a way-point counts as reached inside this radius (Rcyl * 0.05) */
    double waypoints[32 * 3];     /* AuvEnvCyl: x, y, target heading per way-point (verySimpleAuv_cyl.py:33-39) */
    int variant, n_waypoints;
} MvrlAuvParams;

typedef struct MvrlAuvConfig {
    int dtype, max_steps;
    double dt;                 /* 0.02 */
    uint64_t seed, env_id0;
    int auto_reset, stop_on_bounds, apply_noise, device;
} MvrlAuvConfig;

typedef struct MvrlAuvBuffers {
    void* state;        /* T [6][ld] x y psi u v r                                  in/out */
    void* action;       /* T [3][ld]                                                in     */
    void* obs;          /* T [11][ld] dataToState V3, verySimpleAuv.py:201-212      out    */
    void* reward;       /* T [ld]                                                   out    */
    uint8_t* done;      /* [ld]                                                     out    */
    int32_t* istep;     /* [ld]                                                     in/out */
    void* mults;        /* T [11][ld] m I Xuu Yvv Nrr Xu Yv Nr Xact Yact Nact       in (out on reset) */
    void* target;       /* T [2][ld] headingTarget, flowDataTimeOffset              in (out on reset) */
    void* err_o;        /* T [3][ld] perr_o x, perr_o y, herr_o                     in/out */
    void* recent;       /* T [30][ld] the 10 most recent actions (ring)             in/out */
    void* ep_return;    /* T [ld] running episode return                            in/out */
    int32_t* iwp;       /* [ld] way-point index, AuvEnvCyl only (never reset, as upstream)  in/out; nullable for AuvEnv */
    uint32_t* episode;  /* [ld] */
    void* terminal_obs; /* T [11][ld], nullable */
    void* aux;          /* T [14][ld] Fx Fy N Fx_set Fy_set N_set u_current v_current rmsAc r0..r4
                           (log columns of verySimpleAuv.py:389-401); nullable */
    double* ep_stats;   /* [8], nullable */
} MvrlAuvBuffers;

typedef struct MvrlAuv MvrlAuv;

MVRL_API int mvrl_auv_default_params(MvrlAuvParams* out);
MVRL_API int mvrl_auv_create(MvrlAuv** out, const MvrlAuvParams* params, const MvrlAuvConfig* cfg);
MVRL_API int mvrl_auv_destroy(MvrlAuv* h);
/* AuvEnv.reset(applyNoise=...) is a per-call switch upstream (verySimpleAuv.py:216-229): changes whether the NEXT resets (the
 * reset kernel and the step kernel's auto-reset) draw the coefficient / actuation multipliers; takes effect at the next launch. */
MVRL_API int mvrl_auv_set_apply_noise(MvrlAuv* h, int apply_noise);
/* Scaled flow field the env gathers from: device T [nt][ny][nx][nc], nc = 2 (u, v) or 3; the
 * caller keeps it alive.  dx, dy, dt are the SCALED spacings (flowGenerator.py:77-78, 94). */
MVRL_API int mvrl_auv_set_flow(MvrlAuv* h, const void* field, int nt, int ny, int nx, int nc, double dx, double dy, double dt);
MVRL_API int mvrl_auv_step(MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, mvrl_stream_t stream);
/* init nullable T [4][ld]: x, y, heading, headingTarget (fixedInitialValues) */
MVRL_API int mvrl_auv_reset(MvrlAuv* h, int64_t n, int64_t ld, const MvrlAuvBuffers* b, const uint8_t* mask, const void* init,
                            mvrl_stream_t stream);
/* ReconstructedFlow.interp (flowGenerator.py:97-136): t T [n], xy T [2][ld] -> out T [nc][ld] */
MVRL_API int mvrl_flow_interp(int dtype, const void* field, int nt, int ny, int nx, int nc, double dx, double dy, double dt,
                              int64_t n, int64_t ld, const void* t, const void* xy, void* out, mvrl_stream_t stream);
/* ReconstructedFlow.__init__, the SPOD reconstruction (flowGenerator.py:15-23): baseFlowData[t] = Re(modes @ coeffs[:, t]) + lt_mean.
 * modes fp64 [plane][n_modes] and coeffs fp64 [n_modes][nt], each complex (interleaved re, im: numpy complex128) when its
 * *_complex flag is set, else real; mean fp64 [plane]; plane = Ny * Nx * n_fields.  out T [nt][plane] = the [Nt][Ny][Nx][3]
 * base field; accumulation in fp64 whatever T is.  All pointers on one device. */
MVRL_API int mvrl_flow_reconstruct(int dtype, int64_t plane, int n_modes, int nt, const double* modes, int modes_complex,
                                   const double* coeffs, int coeffs_complex, const double* mean, void* out, mvrl_stream_t stream);
/* ReconstructedFlow.scale on the values (flowGenerator.py:80-90): base T [cells][3] -> out T [cells][nc_out] */
MVRL_API int mvrl_flow_scale(int dtype, int64_t cells, const void* base, void* out, int nc_out, double velocityScale,
                             double turbScale, mvrl_stream_t stream);

/* CustomReplayBuffer.add (tag_00.../main_02_sbl_contrib_customBuffer.py:57-160): stores the batch of transitions and its
 * mirror images.  obs / next_obs T [11][ld], act T [3][ld], reward T [n], done [n], timeout [n] or NULL (the
 * "TimeLimit.truncated" flags of the infos, :150-151; NULL = all false) (SoA, as the env holds them) ->
 * buf_obs / buf_next_obs T [buffer_size][n][11], buf_act T [buffer_size][n][3], buf_reward T [buffer_size][n],
 * buf_done, buf_timeout (nullable) [buffer_size][n]; transformation t (0 = identity ... 4) goes to slot
 * (pos + t) % buffer_size, t < n_transforms.  buffer_size counts slots (SB3: transitions // n_envs). */
MVRL_API int mvrl_replay_add_symmetric(int dtype, int64_t n, int64_t ld, const void* obs, const void* next_obs, const void* act,
                                       const void* reward, const uint8_t* done, const uint8_t* timeout, void* buf_obs, void* buf_next_obs,
                                       void* buf_act, void* buf_reward, uint8_t* buf_done, uint8_t* buf_timeout, int64_t buffer_size,
                                       int64_t pos, int n_transforms, mvrl_stream_t stream);

/* ------------------------------------------------------------ rollout actor -- */
/* The policy the reference trains with SB3 (tag_00.../main_00_sbl.py:100-105: MlpPolicy, net_arch [128, 128, 128], GELU)
 * and its Gaussian action head, as one tensor-core kernel on the env's own buffers - BASELINE.json config 5 (rollout
 * collection; the fixed-std head, see below for the SB3 SAC / TQC one): obs float [obs_dim][ld] (the step kernels'
 * structure-of-arrays observation buffer, read in place) ->
 * act float [act_dim][ld] (the structure-of-arrays action buffer the step kernels read).  mean = tanh(W4 gelu(W3 gelu(W2
 * gelu(W1 obs + b1) + b2) + b3) + b4), act = clip(mean + exp(log_std) * eps, -1, 1), eps ~ N(0, 1) from Philox keyed on
 * (seed, env_id0 + i, step) - independent of how the batch is sharded; logp (nullable) [n] = -0.5 sum eps^2 - sum log_std;
 * mean / eps (nullable) [act_dim][ld] for the learner and the tests; deterministic != 0 returns the mean (SB3
 * predict(obs, deterministic=True)).  Operands are bf16 (fp32 accumulate), GELU in its tanh form (torch gelu(approximate=
 * "tanh")).  fp32 only; obs_dim <= 16, act_dim <= 8, hidden width 128.  set_weights takes HOST arrays in torch.nn.Linear layout
 * (W [out][in]) and synchronises; act launches on the caller's stream and does not synchronise.  The kernel is written for the
 * sm_100a tensor core (tcgen05.mma from shared-memory descriptors, accumulators in tensor memory; one CTA per SM takes all 512
 * TMEM columns while it runs); MVRL_POLICY_MMA_SYNC=1 in the environment of mvrl_policy_create selects the warp-level mma.sync
 * implementation of the same network instead (same noise bit for bit, means within the fp32 summation order).
 *
 * Two action heads, chosen at create time:
 *   MVRL_POLICY_HEAD_FIXED_STD (mvrl_policy_create): the head described above - a generic head with one state-independent
 *     log_std vector, tanh before the noise and no Jacobian or 2 pi term in logp.  It is NOT the head SB3 trains.
 *   MVRL_POLICY_HEAD_SQUASHED: the Actor of SB3 SAC / sb3_contrib TQC (SquashedDiagGaussianDistribution).  Two head layers,
 *     mu = W_mu h + b_mu and log_std = clamp(W_log_std h + b_log_std, -20, 2), a = tanh(mu + exp(log_std) * eps),
 *     logp = sum(-eps^2 / 2 - log_std - log(2 pi) / 2) - sum log(1 - a^2 + 1e-6), the log-prob of a.  With noise_std set,
 *     act = clip(a + noise_std * xi, -1, 1), xi ~ N(0, 1) from its own Philox stream keyed like eps (SB3's NormalActionNoise
 *     of off-policy collection; eps does not change with it, logp stays that of a); without it act = a.  deterministic != 0
 *     gives act = tanh(mu), no noise.  mean = mu (before tanh, SB3's mean_actions); log_std (nullable) [act_dim][ld].  Same
 *     bf16 operands and tanh-form GELU as above.
 * mvrl_policy_set_weights / _set_weights_squashed serve the fixed / squashed head (MVRL_EINVAL for the other kind, also for
 * an unknown head and for a log_std output on a fixed handle); mvrl_policy_act is mvrl_policy_act_ex with log_std = NULL.
 *
 * Weight sync.  One kernel (policy_pack_kernel) packs every parameter block of a handle from fp32 arrays in device memory.
 * The host entries (set_weights, _set_weights_squashed) copy their host arrays into a staging buffer the handle owns, run it
 * on the legacy default stream and synchronise.  mvrl_policy_set_weights_squashed_device reads a learner's CUDA tensors in
 * place and packs on the caller's stream without synchronising, so a collect / learn loop can sync after every gradient step
 * and be captured as a CUDA graph.  The fixed head has no device entry, on purpose: its std = expf(log_std) and
 * logp = -sum(log_std) are computed on the host and reach the kernels as launch arguments, so a stream-ordered path would
 * change every fixed-head act kernel and the rounding of std (glibc's expf and a device exp differ in the last bit for some
 * inputs); it is the generic head, not the one SB3 trains.
 *
 * Two numeric precisions, chosen at create time (mvrl_policy_create_ex; mvrl_policy_create / _create_head give BF16), both
 * heads, same set_weights / act calls:
 *   MVRL_POLICY_PRECISION_BF16: the kernels described above - bf16 operands, tanh-form GELU, tanh.approx for the fixed
 *     head's mean.  mu / log_std within ~4e-3 of SB3's fp32 network (measured on a B200, DESIGN.md K7).  The fast mode.
 *   MVRL_POLICY_PRECISION_FP32: the network SB3 evaluates - fp32 operands as split bf16 (hi + lo, three tensor-core products
 *     per layer: A_hi B_hi + A_lo B_hi + A_hi B_lo), GELU in its erf form (torch.nn.GELU()), tanhf for the fixed head's
 *     mean; within 5e-5 * max(1, |ref|) of the fp64 network (measured: DESIGN.md K7).  Same Philox streams, eps, action
 *     noise, clamp and log-prob as BF16: the same seed gives the same eps bit for bit.  It has one implementation (tcgen05):
 *     MVRL_POLICY_MMA_SYNC=1 applies to BF16 handles only, and creating an FP32 handle with it set is MVRL_EINVAL.
 * An unknown precision is MVRL_EINVAL. */
#define MVRL_POLICY_HEAD_FIXED_STD 0   /* the existing head (generic, not SB3's) */
#define MVRL_POLICY_HEAD_SQUASHED 1    /* SB3 SAC / sb3_contrib TQC Actor */
#define MVRL_POLICY_PRECISION_BF16 0   /* the existing kernels: bf16 operands, tanh-form GELU (default) */
#define MVRL_POLICY_PRECISION_FP32 1   /* split-bf16 tensor-core products, erf GELU: SB3's fp32 network */
typedef struct MvrlPolicy MvrlPolicy;
MVRL_API int mvrl_policy_create(MvrlPolicy** out, int device, int obs_dim, int act_dim);
MVRL_API int mvrl_policy_create_head(MvrlPolicy** out, int device, int obs_dim, int act_dim, int head);
MVRL_API int mvrl_policy_create_ex(MvrlPolicy** out, int device, int obs_dim, int act_dim, int head, int precision);
MVRL_API int mvrl_policy_destroy(MvrlPolicy* h);
MVRL_API int mvrl_policy_set_weights(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                     const float* W3, const float* b3, const float* W4, const float* b4, const float* log_std);
/* HOST arrays in torch.nn.Linear layout (W_mu, W_log_std [act_dim][128]); noise_std [act_dim] (finite, >= 0) or NULL = no
 * action noise.  Synchronises, like mvrl_policy_set_weights. */
MVRL_API int mvrl_policy_set_weights_squashed(MvrlPolicy* h, const float* W1, const float* b1, const float* W2, const float* b2,
                                              const float* W3, const float* b3, const float* W_mu, const float* b_mu,
                                              const float* W_log_std, const float* b_log_std, const float* noise_std);
/* DEVICE arrays (fp32, torch.nn.Linear layout, on the handle's device); noise_std a HOST array [act_dim] or NULL, as in
 * mvrl_policy_set_weights_squashed.  Packs on `stream`, does not synchronise, capturable in a CUDA graph: an act launched
 * on the same stream afterwards sees the new weights, one queued before sees the old; an act on another stream must be
 * ordered by the caller (event / wait_stream).  MVRL_EINVAL for a null argument, a fixed-head handle, a negative or
 * non-finite noise_std, and a weight pointer that is not device memory on the handle's device. */
MVRL_API int mvrl_policy_set_weights_squashed_device(MvrlPolicy* h, const float* W1, const float* b1, const float* W2,
        const float* b2, const float* W3, const float* b3, const float* W_mu, const float* b_mu, const float* W_log_std,
        const float* b_log_std, const float* noise_std, mvrl_stream_t stream);
MVRL_API int mvrl_policy_act(MvrlPolicy* h, int64_t n, int64_t ld, const float* obs, float* act, float* logp, float* mean,
                             float* eps, uint64_t seed, uint64_t env_id0, uint32_t step, int deterministic, mvrl_stream_t stream);
MVRL_API int mvrl_policy_act_ex(MvrlPolicy* h, int64_t n, int64_t ld, const float* obs, float* act, float* logp, float* mean,
                                float* log_std, float* eps, uint64_t seed, uint64_t env_id0, uint32_t step, int deterministic,
                                mvrl_stream_t stream);

/* ------------------------------------------------------------ calibration -- */
/* K6: measured FMA throughput of the FP32 / FP64 pipe in TFLOP/s (2 flop per FMA,
 * 8 independent chains per thread, 8 x 256 threads per SM).  Roofline denominator
 * for the FP-pipe-bound step kernels; synchronises (measurement utility). */
MVRL_API int mvrl_measure_fma_peak(int dtype, int device, int iters, double* tflops_out, double* ms_out);

#ifdef __cplusplus
}
#endif
#endif /* MVRL_H_ */
