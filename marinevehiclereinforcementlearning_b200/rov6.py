"""Batched BlueROV2 Heavy 6DoF engine: host-side owner of the device buffers
and of the libmvrl handle.  All numerics run in the CUDA kernels behind the C
ABI (include/mvrl.h); this module only allocates torch tensors, marshals
pointers and mirrors the reference's attribute names.

Reference surface mirrored: dynamicsModel_BlueROV2_Heavy_6DoF.py:75-218
(vehicle constants), :445-594 (env reset/step semantics).
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _lib
from ._envbase import _HandleCache, _VecEnv, _Versioned
from ._lib import ACT_FORCE, ACT_RPM, ACT_SETPOINT

ACTION_MODES = {"rpm": ACT_RPM, "force": ACT_FORCE, "setpoint": ACT_SETPOINT, "pid": ACT_SETPOINT,
                ACT_RPM: ACT_RPM, ACT_FORCE: ACT_FORCE, ACT_SETPOINT: ACT_SETPOINT}
ACTION_DIM = {ACT_RPM: 8, ACT_FORCE: 6, ACT_SETPOINT: 6}

# 6DoF.py:46-54
PID6_DEFAULTS = dict(
    windup=[2., 2., 2., 90. / 180. * np.pi, 90. / 180. * np.pi, 90. / 180. * np.pi],
    max=[50., 50., 50., 1., 1., 2.],
    Kp=[25., 25., 25., 10., 10., 1.],
    Ki=[2., 2., 2., 0.1, 0.1, 0.2],
    Kd=[20., 20., 20., 5., 5., 0.65])


class Rov6Constants(_Versioned):
    """Vehicle constants with the reference's attribute names
    (6DoF.py:83-218).  Pure host-side set-up, done once per vehicle exactly as
    the reference does in ``__init__`` (numpy ``pinv`` for the allocation so the
    matrices are bit-identical to the reference's)."""

    def __init__(self):
        self.rho_f = 1000.
        self.m = 11.4
        self.dispVol = self.m / self.rho_f
        self.Length = 0.457
        self.Width = 0.338
        self.CB = np.array([0., 0., 0.])
        self.CG = np.array([0., 0., 0.05])
        self.I = np.array([[0.16, 0., 0.], [0., 0.16, 0.], [0., 0., 0.16]])
        self.x_origin = np.array([0., 0., 0.0375])
        self.Xudot, self.Yvdot, self.Zwdot = -5.5, -12.7, -14.57
        self.Kpdot = self.Mqdot = self.Nrdot = -0.12
        self.Yrdot = self.Zvdot = self.Nvdot = 0.
        self.Xuu, self.Yvv, self.Zww = -18.18, -21.66, -36.99
        self.Kpp = self.Mqq = self.Nrr = -1.55
        self.Yrr = self.Ypp = self.Zqq = self.Kvv = self.Krr = 0.
        self.Mww = -1.55
        self.Nvv = self.Npp = 0.
        self.Xu, self.Yv, self.Zw = -4.03, -6.22, -5.18
        self.Kp = self.Mq = self.Nr = -0.07
        self.Yr = self.Yp = self.Zq = self.Kv = self.Kr = self.Mw = self.Nv = self.Np = 0.
        self.D_thruster = 0.1
        self.alphaThruster = 33. / 180. * np.pi
        self.l_x, self.l_y, self.l_z = 0.1475, 0.101, 0.068
        self.l_x_v, self.l_y_v, self.l_z_v = 0.120, 0.22, 0.0
        self.Kt_thruster = 40. / (1000. * (3500. / 60.) ** 2. * self.D_thruster ** 4.)
        a = self.alphaThruster
        self.thrusterPositions = np.array([
            [self.l_x, self.l_y, self.l_z], [self.l_x, -self.l_y, self.l_z],
            [-self.l_x, self.l_y, self.l_z], [-self.l_x, -self.l_y, self.l_z],
            [self.l_x_v, self.l_y_v, self.l_z_v], [self.l_x_v, -self.l_y_v, self.l_z_v],
            [-self.l_x_v, self.l_y_v, self.l_z_v], [-self.l_x_v, -self.l_y_v, self.l_z_v]])
        self.thrusterNormals = np.array([
            [np.cos(a), -np.sin(a), 0.], [np.cos(a), np.sin(a), 0.],
            [-np.cos(a), -np.sin(a), 0.], [-np.cos(a), np.sin(a), 0.],
            [0., 0., -1.], [0., 0., 1.], [0., 0., 1.], [0., 0., -1.]])
        from .resources import computeThrustAllocation
        self.A, self.Ainv = computeThrustAllocation(self.thrusterPositions, self.thrusterNormals)
        self.disableThrusters = False
        self.rpmMax = 3500.
        self.rpmDeadband = 300.
        self.pid = {k: np.array(v, dtype=float) for k, v in PID6_DEFAULTS.items()}

    def massMatrix(self):
        """Mrb + Ma as assembled at 6DoF.py:286-299 (Ma[2,2] = -Zvdot)."""
        m, (xg, yg, zg) = self.m, self.CG
        M = np.array([
            [m, 0., 0., 0., m * zg, -m * yg],
            [0., m, 0., -m * zg, 0., m * xg],
            [0., 0., m, m * yg, -m * xg, 0.],
            [0., -m * zg, m * yg, 0., 0., 0.],
            [m * zg, 0., -m * xg, 0., 0., 0.],
            [-m * yg, m * xg, 0., 0., 0., 0.]])
        M[3:, 3:] = self.I
        return M + -1. * np.diag([self.Xudot, self.Yvdot, self.Zvdot, self.Kpdot, self.Mqdot, self.Nrdot])

    def to_struct(self):
        p = _lib.MvrlRov6Params()
        p.rho_f, p.m, p.Length = self.rho_f, self.m, self.Length
        p.CG[:] = list(map(float, self.CG))
        p.CB[:] = list(map(float, self.CB))
        p.I[:] = list(map(float, np.asarray(self.I).reshape(-1)))
        for name in ("Xudot", "Yvdot", "Zwdot", "Kpdot", "Mqdot", "Nrdot",
                     "Xu", "Yv", "Yp", "Yr", "Zw", "Zq", "Kv", "Kp", "Kr", "Mw", "Mq", "Nv", "Np", "Nr",
                     "Xuu", "Yvv", "Ypp", "Yrr", "Zww", "Zqq", "Kvv", "Kpp", "Krr", "Mww", "Mqq", "Nvv", "Npp", "Nrr"):
            setattr(p, name, float(getattr(self, name)))
        p.W = self.m * 9.81                                   # 6DoF.py:374
        p.B = self.dispVol * self.rho_f * 9.81                # 6DoF.py:375
        p.thrust_coef = self.rho_f * self.D_thruster ** 4. * self.Kt_thruster
        p.rpm_max, p.rpm_deadband = self.rpmMax, self.rpmDeadband
        M = self.massMatrix()
        p.M[:] = list(M.reshape(-1))
        p.Minv[:] = list(np.linalg.inv(M).reshape(-1))
        p.A[:] = list(np.asarray(self.A, dtype=float).reshape(-1))
        p.Ainv[:] = list(np.asarray(self.Ainv, dtype=float).reshape(-1))
        p.pid_Kp[:] = list(self.pid["Kp"]); p.pid_Ki[:] = list(self.pid["Ki"]); p.pid_Kd[:] = list(self.pid["Kd"])
        p.pid_windup[:] = list(self.pid["windup"]); p.pid_max[:] = list(self.pid["max"])
        p.disable_thrusters = 1 if self.disableThrusters else 0
        return p


class _RovHandle(_lib.Handle):
    """An opaque ``MvrlRov6*`` / ``MvrlRov3*`` (``PREFIX``) of the given constants and configuration."""

    def __init__(self, consts, dtype, action_mode, n_sub=8, dt=0.2, max_steps=250, seed=0, env_id0=0,
                 auto_reset=False, fixed_sp=False, device=0, fast_math=False):
        self.cfg = _lib.MvrlRov6Config(
            dtype=_lib.torch_dtype_code(dtype), action_mode=ACTION_MODES[action_mode], n_sub=int(n_sub),
            max_steps=int(max_steps), dt=float(dt), seed=int(seed) & (2 ** 64 - 1), env_id0=int(env_id0),
            auto_reset=int(bool(auto_reset)), fixed_sp=int(bool(fixed_sp)), device=int(device), fast_math=int(bool(fast_math)))
        self.params = consts.to_struct()
        super().__init__(self.PREFIX, C.byref(self.params), C.byref(self.cfg))


class Rov6Handle(_RovHandle):
    PREFIX = "mvrl_rov6"

    @property
    def specialised(self):
        return bool(self.lib.mvrl_rov6_is_specialised(self._h))

    @property
    def specialisation(self):
        """0 = generic kernels, 1 = default-sparsity kernels, 2 = default vehicle: fp32 kernels with compile-time constants."""
        return int(self.lib.mvrl_rov6_is_specialised(self._h))


def _device_index(device):
    _lib.require_cuda()
    d = torch.device(device)
    if d.type != "cuda":
        raise RuntimeError("the batched simulator runs on CUDA devices only (got %s); there is no CPU fallback" % d)
    return d.index if d.index is not None else torch.cuda.current_device()


class _RovVecEnv(_VecEnv):
    """The 6DoF and 3DoF batched envs: semantics per environment are those of
    the reference's Gym env with the integrator fixed to classic RK4 x ``n_sub``."""
    STATE_DIM, OBS_DIM, SP_DIM, PATH_DIM, CTRL_DIM, AUX_DIM = 12, 9, 6, 6, 13, 14
    ACTION_DIM = {ACT_RPM: 8, ACT_FORCE: 6, ACT_SETPOINT: 6}
    BUFFERS = _lib.MvrlRov6Buffers
    _STATE_KEYS = ("_state", "_istep", "_setpoint", "_path", "_ctrl", "_episode", "_obs", "fixedSp")

    def __init__(self, num_envs, seed=0, dt=0.2, maxSteps=250, n_sub=8, action_mode="setpoint",
                 dtype=torch.float32, device="cuda", auto_reset=True, env_id0=0, fast_math=False,
                 record_aux=False, record_terminal_obs=True, collect_stats=True, vehicle=None):
        self.n_sub = int(n_sub)
        self.action_mode = ACTION_MODES[action_mode]
        if self.action_mode not in self.ACTION_DIM:
            raise ValueError("action_mode %r is not supported by %s" % (action_mode, type(self).__name__))
        self.fast_math = bool(fast_math)
        self.vehicle = vehicle if vehicle is not None else self.CONSTANTS()
        self.lenAction = self.ACTION_DIM[self.action_mode]
        self.fixedSp = False
        super().__init__(self.HANDLE.PREFIX, num_envs, torch.device("cuda", _device_index(device)), dtype, dt, maxSteps, seed,
                         env_id0, auto_reset, record_aux, record_terminal_obs, collect_stats)

    def _extra_buffers(self):
        self._setpoint, self._path, self._ctrl = self._zeros(self.SP_DIM), self._zeros(self.PATH_DIM), self._zeros(self.CTRL_DIM)

    # -- handle management (re-created when a constant or a flag changes) ----
    def _get_handle(self):
        return self._cached_handle((self.vehicle.fingerprint(), self.fixedSp, self.auto_reset, self.n_sub, self.dt,
                                    self._max_episode_steps, self.seed, self.env_id0, self.fast_math, self.action_mode))

    def _new_handle(self):
        return self.HANDLE(self.vehicle, self.dtype, self.action_mode, n_sub=self.n_sub, dt=self.dt,
                           max_steps=self._max_episode_steps, seed=self.seed, env_id0=self.env_id0,
                           auto_reset=self.auto_reset, fixed_sp=self.fixedSp, device=self.device.index,
                           fast_math=self.fast_math)

    # -- views -----------------------------------------------------------------
    @property
    def systemState(self):
        return self._state[:, :self.num_envs].T

    @property
    def setPoint(self):
        return self._setpoint[:, :self.num_envs].T

    @property
    def path(self):
        """[N, 2, dims] way-points (6DoF.py:497, 509 / 3DoF.py:423, 435)."""
        return self._path[:, :self.num_envs].T.reshape(self.num_envs, 2, self.PATH_DIM // 2)

    def reset(self, initialSetpoint=None, mask=None):
        """6DoF.py:485-529 / 3DoF.py:411-453.  ``initialSetpoint=None`` takes the
        random branch (for 6DoF defined here; the reference's own line raises -
        see DESIGN.md)."""
        self.fixedSp = initialSetpoint is not None
        h = self._get_handle()
        m = self._begin_reset(mask)
        sp = None
        if initialSetpoint is not None:
            vals = [float(v) for v in np.asarray(initialSetpoint, dtype=float).reshape(self.SP_DIM)]
            sp = (C.c_double * self.SP_DIM)(*vals)
        _lib.check(h.fn("reset")(h._h, self.num_envs, self.ld, C.byref(self._bufs), _lib.ptr(m), sp,
                                 _lib.current_stream(self.device)))
        return self.state

    def observe(self):
        """dataToState for the current device state (6DoF.py:467-483 / 3DoF.py:397-409),
        [N, obs]: resources.angleError / clip run on the device through torch views of the
        same SoA buffers the kernels use."""
        from . import resources
        n, L3 = self.num_envs, self.vehicle.Length * 3.
        half = self.PATH_DIM // 2
        pos = self._state[:half, :n]
        ang_sp = self._setpoint[half:, :n]
        ang = self._state[half:self.SP_DIM, :n]
        err = torch.stack([resources.angleError(ang_sp[k].contiguous(), ang[k].contiguous()) for k in range(ang.shape[0])])
        obs = torch.cat([(self._path[:half, :n] - pos) / L3, (self._path[half:, :n] - pos) / L3, err / (45. / 180. * np.pi)])
        return obs.clamp(-1., 1.).T


class BlueROV2Heavy6DoFVecEnv(_RovVecEnv):
    """Batched ``BlueROV2Heavy6DoFEnv`` (6DoF.py:445-594): 12 states, 9
    observations; actions per ``action_mode``: "setpoint" (reference Gym
    semantics, 6 in [-1, 1]), "force" (6 earth-frame generalised forces) or
    "rpm" (8 thruster rpm)."""
    HANDLE, CONSTANTS = Rov6Handle, Rov6Constants
    HISTORY_COLUMNS = (["t"] + ["x", "y", "z", "phi", "theta", "psi"] + ["u", "v", "w", "p", "q", "r"]
                       + ["F%d" % i for i in range(6)] + ["u%d" % i for i in range(8)]
                       + ["x_d", "y_d", "z_d", "phi_d", "theta_d", "psi_d"])  # 6DoF.py:584-587

    def step_host(self, actions, obs_out=None, reward_out=None, done_out=None, chunks=0):
        """One env step for a caller that lives on the HOST: ``actions`` is a CPU tensor
        ``[N, A]`` (pinned memory lets the copies overlap), results land in CPU tensors
        ``obs [N, obs]``, ``reward [N]``, ``done [N]`` (uint8), allocated pinned on first use.
        Runs ``mvrl_rov6_step_host``: upload, SoA transpose, fused step, transpose back and
        download are pipelined over ``chunks`` equal pieces of the batch (0: the library's
        default).  Returns when the host tensors are complete."""
        n = self.num_envs
        if actions.device.type != "cpu" or actions.dtype != self.dtype or tuple(actions.shape) != (n, self.lenAction) or not actions.is_contiguous():
            raise ValueError("actions must be a contiguous CPU tensor [%d, %d] of %s" % (n, self.lenAction, self.dtype))
        if obs_out is None:
            if getattr(self, "_h_obs", None) is None:
                self._h_obs = torch.empty((n, self.lenObs), dtype=self.dtype).pin_memory()
                self._h_reward = torch.zeros(n, dtype=self.dtype).pin_memory()   # reward == 0 (6DoF.py:575): never shipped over PCIe
                self._h_done = torch.empty(n, dtype=torch.uint8).pin_memory()
            obs_out, reward_out, done_out = self._h_obs, self._h_reward, self._h_done
        elif reward_out is not None:
            reward_out.zero_()   # caller-owned array: the library zero-fills it only when it captures the pipeline
        h = self._get_handle()
        self._bufs.action = self._action.data_ptr()
        _lib.check(h.lib.mvrl_rov6_step_host(h._h, n, self.ld, C.byref(self._bufs), C.c_void_p(actions.data_ptr()),
                                             C.c_void_p(obs_out.data_ptr()),
                                             None if reward_out is None else C.c_void_p(reward_out.data_ptr()),
                                             None if done_out is None else C.c_void_p(done_out.data_ptr()),
                                             int(chunks), _lib.current_stream(self.device)))
        return obs_out, reward_out, done_out

    def step_range_async(self, first, count):
        """Launch the fused step for environments ``[first, first + count)`` only (``mvrl_rov6_step_range``)."""
        h = self._get_handle()
        _lib.check(h.lib.mvrl_rov6_step_range(h._h, int(first), int(count), self.ld, C.byref(self._bufs), _lib.current_stream(self.device)))


class _RovDerivs(_HandleCache):
    """Batched ``derivs`` of the vehicle of ``HANDLE`` and ``CONSTANTS``: ``ctrl`` has ``CTRL_ROWS`` rows, the aux
    output ``AUX_ROWS``."""

    def __init__(self, consts=None, dtype=torch.float64, action_mode="rpm", device="cuda"):
        self.consts = consts if consts is not None else self.CONSTANTS()
        self.dtype, self.action_mode = dtype, ACTION_MODES[action_mode]
        self.device = torch.device("cuda", _device_index(device))

    def _get_handle(self):
        return self._cached_handle(self.consts.fingerprint())

    def _new_handle(self):
        return self.HANDLE(self.consts, self.dtype, self.action_mode, device=self.device.index)

    @classmethod
    def new_ctrl(cls, n, dtype=torch.float64, device="cuda"):
        """Fresh PID state (6DoF.py:37-41): eOld=None (NaN marker), eInt=0, tOld=0."""
        c = torch.zeros((cls.CTRL_ROWS, n), dtype=dtype, device=device)
        c[0] = float("nan")
        return c

    def __call__(self, state, act=None, t=None, setpoint=None, ctrl=None, want_aux=False):
        h = self._get_handle()
        prep = lambda x: None if x is None else x.to(device=self.device, dtype=self.dtype).contiguous()
        state, act, t, setpoint = prep(state), prep(act), prep(t), prep(setpoint)
        if ctrl is not None and (ctrl.dtype != self.dtype or not ctrl.is_contiguous() or ctrl.device != self.device):
            raise ValueError("ctrl must be a contiguous [%d, N] tensor of the model dtype on the model device" % self.CTRL_ROWS)
        n = state.shape[1]
        dstate = torch.empty_like(state)
        aux = torch.empty((self.AUX_ROWS, n), dtype=self.dtype, device=self.device) if want_aux else None
        _lib.check(h.fn("derivs")(h._h, n, n, _lib.ptr(state), _lib.ptr(act), _lib.ptr(t), _lib.ptr(setpoint),
                                  _lib.ptr(ctrl), _lib.ptr(dstate), _lib.ptr(aux), _lib.current_stream(self.device)))
        return (dstate, aux) if want_aux else dstate


class Rov6Derivs(_RovDerivs):
    """Batched ``BlueROV2Heavy6DoF.derivs`` (6DoF.py:406-442): one derivative
    evaluation per environment through ``mvrl_rov6_derivs`` (kernel K2).

    Feature-major tensors: ``state`` [12, N]; ``act`` [8, N] rpm or [6, N]
    earth-frame forces; set-point mode takes ``t`` [N], ``setpoint`` [6, N] and
    the controller state ``ctrl`` [13, N] (updated in place like the reference
    mutates its controller)."""
    HANDLE, CONSTANTS, CTRL_ROWS, AUX_ROWS = Rov6Handle, Rov6Constants, 13, 50
