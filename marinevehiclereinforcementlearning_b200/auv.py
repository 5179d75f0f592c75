"""Batched legacy "verySimpleAuv" engine (kernel K4) and the turbulence field
it gathers from.  Host side only: owns the torch tensors and the libmvrl
handle; every number comes from the CUDA kernels behind ``mvrl_auv_*`` /
``mvrl_flow_*`` (include/mvrl.h).

Reference surface mirrored:
tag_00_Dec2023_simpleControlTurbulence/verySimpleAuv.py:76-410 (AuvEnv) and
tag_00_Dec2023_simpleControlTurbulence/flowGenerator.py:13-159
(ReconstructedFlow.scale / interp / interpField).
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._envbase import _VecEnv
from .rov6 import _device_index

# log columns written by the step kernel next to state / obs (verySimpleAuv.py:389-401)
AUX_COLUMNS = ("Fx", "Fy", "N", "Fx_set", "Fy_set", "N_set", "u_current", "v_current", "rmsAc", "r0", "r1", "r2", "r3", "r4")


class FlowField:
    """Device-resident turbulence field ``[Nt, Ny, Nx, 3]`` (u/Uinf, v/Uinf, Cp)
    on a uniform grid, with ``ReconstructedFlow.scale`` and ``.interp`` running
    as CUDA kernels (``mvrl_flow_scale`` / ``mvrl_flow_interp``).

    The SPOD reconstruction of ``ReconstructedFlow.__init__``
    (flowGenerator.py:15-23) needs ``coeffs.npy`` / ``modes_r.npy`` which are
    absent from the reference checkout, so the base field is supplied by the
    caller (a reconstructed one, or the synthetic mean + noise field of
    SURVEY.md 8(d) config 4)."""

    def __init__(self, baseFlowData, baseDx=0.005, baseDy=0.005, baseDt=0.002, baseCoords=None, dtype=torch.float32, device="cuda"):
        self.device = torch.device("cuda", _device_index(device))
        self.dtype = dtype
        base = torch.as_tensor(baseFlowData)
        if base.dim() != 4 or base.shape[3] != 3:
            raise ValueError("baseFlowData must be [Nt, Ny, Nx, 3] (u/Uinf, v/Uinf, Cp), got %s" % (tuple(base.shape),))
        self.baseFlowData = base.to(device=self.device, dtype=dtype).contiguous()
        self.baseDx, self.baseDy, self.baseDt = float(baseDx), float(baseDy), float(baseDt)
        nt, ny, nx, _ = self.baseFlowData.shape
        if baseCoords is None:  # uniform grid starting at the origin, (y, x) orientation like the reference
            xs, ys = np.arange(nx) * self.baseDx, np.arange(ny) * self.baseDy
            baseCoords = np.stack(np.meshgrid(xs, ys), axis=2)
        self.baseCoords = np.asarray(baseCoords, dtype=float)
        self.baseTime = np.arange(nt) * self.baseDt
        self.flowData = torch.empty_like(self.baseFlowData)
        self._uv = torch.empty((nt, ny, nx, 2), dtype=dtype, device=self.device)
        self.scale(1., 1., 1.)

    @property
    def shape(self):
        return tuple(self.baseFlowData.shape)

    def scale(self, sizeScale, velocityScale, turbScale, translate=(0, 0)):
        """flowGenerator.py:53-95.  Fills ``flowData`` (3 fields) and the 2-field
        (u, v) copy the env kernel gathers from.  ``translate`` only moves
        ``coords``; ``interp`` ignores it exactly like the reference."""
        lib = _lib.load()
        self.coords = self.baseCoords.copy() * sizeScale + translate
        self.dx = self.baseDx * sizeScale
        self.dy = self.baseDy * sizeScale
        cells = self.baseFlowData.numel() // 3
        code = _lib.torch_dtype_code(self.dtype)
        s = _lib.current_stream(self.device)
        _lib.check(lib.mvrl_flow_scale(code, cells, _lib.ptr(self.baseFlowData), _lib.ptr(self.flowData), 3, float(velocityScale), float(turbScale), s))
        _lib.check(lib.mvrl_flow_scale(code, cells, _lib.ptr(self.baseFlowData), _lib.ptr(self._uv), 2, float(velocityScale), float(turbScale), s))
        self.dt = self.baseDt * sizeScale / max(1e-6, velocityScale)
        self.time = np.array([i * self.dt for i in range(self.shape[0])])

    def interp(self, time, xy):
        """flowGenerator.py:97-136.  Scalars / numpy (``time`` float, ``xy`` 2-vector) ->
        numpy ``(3,)`` like the reference; tensors ``time [N]``, ``xy [N, 2]`` -> ``[N, 3]`` on the device."""
        lib = _lib.load()
        batched = isinstance(time, torch.Tensor) or isinstance(xy, torch.Tensor)
        t = torch.as_tensor(time, dtype=self.dtype, device=self.device).reshape(-1).contiguous()
        p = torch.as_tensor(xy, dtype=self.dtype, device=self.device).reshape(-1, 2).T.contiguous()  # [2, N]
        n = t.numel()
        if p.shape[1] != n:
            raise ValueError("time and xy disagree on the number of points")
        out = torch.empty((3, n), dtype=self.dtype, device=self.device)
        nt, ny, nx, _ = self.shape
        _lib.check(lib.mvrl_flow_interp(_lib.torch_dtype_code(self.dtype), _lib.ptr(self.flowData), nt, ny, nx, 3, self.dx, self.dy, self.dt,
                                        n, n, _lib.ptr(t), _lib.ptr(p), _lib.ptr(out), _lib.current_stream(self.device)))
        if batched:
            return out.T
        res = out.T.cpu().numpy().astype(float)
        return res[0] if np.ndim(time) == 0 else res

    def interpField(self, time):
        """flowGenerator.py:138-159: the whole plane interpolated in time only ->
        ``[Ny, Nx, 3]``; evaluated by ``mvrl_flow_interp`` at every grid node."""
        nt, ny, nx, _ = self.shape
        jj, ii = torch.meshgrid(torch.arange(ny, device=self.device), torch.arange(nx, device=self.device), indexing="ij")
        xy = torch.stack([ii.reshape(-1).to(self.dtype) * self.dx, jj.reshape(-1).to(self.dtype) * self.dy], dim=1)
        t = torch.full((ny * nx,), float(time), dtype=self.dtype, device=self.device)
        return self.interp(t, xy).reshape(ny, nx, 3)


class AuvVecEnv(_VecEnv):
    """N legacy ``AuvEnv`` environments stepped by one fused CUDA kernel
    (verySimpleAuv.py:264-410): trilinear flow gather, explicit Euler step, V3
    observation, shaped reward with the 10-deep action ring, bounds
    termination and SB3-style auto-reset."""
    STATE_DIM, OBS_DIM, ACT_DIM, AUX_DIM = 6, 11, 3, len(AUX_COLUMNS)
    VARIANT = _lib.AUV_PLAIN
    BOUNDS = 1.
    PREFIX = "mvrl_auv"
    BUFFERS = _lib.MvrlAuvBuffers
    _STATE_KEYS = ("_state", "_istep", "_mults", "_target", "_err_o", "_recent", "_ep_return", "_iwp", "_episode", "_obs")
    # verySimpleAuv.py:389-401
    HISTORY_COLUMNS = (["step", "time", "reward", "x", "y", "psi", "x_d", "y_d", "psi_d"]
                       + ["Fx", "Fy", "N", "Fx_set", "Fy_set", "N_set"]
                       + ["u", "v", "r", "u_current", "v_current", "rmsAc"]
                       + ["r%d" % i for i in range(5)] + ["a%d" % i for i in range(3)] + ["s%d" % i for i in range(11)])

    def __init__(self, num_envs, flow, seed=0, dt=0.02, maxSteps=250, noiseMagCoeffs=0.0, noiseMagActuation=0.0,
                 stopOnBoundsExceeded=True, applyNoise=True, dtype=torch.float32, device=None, auto_reset=True,
                 env_id0=0, record_aux=False, record_terminal_obs=True, collect_stats=True):
        self.flow = flow
        device = flow.device if device is None else torch.device("cuda", _device_index(device))
        if flow.device != device or flow.dtype != dtype:
            raise ValueError("the flow field must live on the env's device with the env's dtype")
        self.stopOnBoundsExceeded, self.applyNoise = bool(stopOnBoundsExceeded), bool(applyNoise)
        # verySimpleAuv.py:110-132
        self.xMinMax, self.yMinMax = [-self.BOUNDS, self.BOUNDS], [-self.BOUNDS, self.BOUNDS]
        self.waypoints, self.wpThreshold = np.zeros((0, 3)), 0.
        self.m, self.Izz = 11.4, 0.16
        self.Xuu, self.Yvv, self.Nrr = -18.18 * 2.21, -21.66 * 4.87, -1.55
        self.Xu, self.Yv, self.Nr = -4.03 * 2.21, -6.22 * 4.87, -0.07
        self.maxForce, self.maxMoment = 150., 20.
        self.noiseMagCoeffs, self.noiseMagActuation = float(noiseMagCoeffs), float(noiseMagActuation)
        self.lenAction = self.ACT_DIM
        super().__init__(self.PREFIX, num_envs, device, dtype, dt, maxSteps, seed, env_id0, auto_reset, record_aux,
                         record_terminal_obs, collect_stats)

    def _extra_buffers(self):
        z = self._zeros
        self._mults, self._target, self._err_o, self._recent = z(11), z(2), z(3), z(30)
        self._mults.fill_(1.)
        self._ep_return = z()
        self._iwp = z(dtype=torch.int32)       # AuvEnvCyl only; never reset, as upstream

    def _get_handle(self):
        f = self.flow
        return self._cached_handle((
            self.m, self.Izz, self.Xuu, self.Yvv, self.Nrr, self.Xu, self.Yv, self.Nr, self.maxForce, self.maxMoment,
            tuple(self.xMinMax), tuple(self.yMinMax), self.noiseMagCoeffs, self.noiseMagActuation, self.dt,
            self._max_episode_steps, self.seed, self.env_id0, self.auto_reset, self.stopOnBoundsExceeded, self.applyNoise,
            f._uv.data_ptr(), f.dx, f.dy, f.dt, self.wpThreshold, np.asarray(self.waypoints, dtype=float).tobytes()))

    def _new_handle(self):
        p = _lib.MvrlAuvParams(m=self.m, Izz=self.Izz, Xuu=self.Xuu, Yvv=self.Yvv, Nrr=self.Nrr, Xu=self.Xu, Yv=self.Yv, Nr=self.Nr,
                               maxForce=self.maxForce, maxMoment=self.maxMoment, xMin=self.xMinMax[0], xMax=self.xMinMax[1],
                               yMin=self.yMinMax[0], yMax=self.yMinMax[1], noiseMagCoeffs=self.noiseMagCoeffs,
                               noiseMagActuation=self.noiseMagActuation, wp_threshold=float(self.wpThreshold),
                               variant=self.VARIANT, n_waypoints=len(self.waypoints))
        flat = np.asarray(self.waypoints, dtype=float).reshape(-1)
        p.waypoints[:len(flat)] = list(flat)
        cfg = _lib.MvrlAuvConfig(dtype=_lib.torch_dtype_code(self.dtype), max_steps=self._max_episode_steps, dt=self.dt,
                                 seed=self.seed & (2 ** 64 - 1), env_id0=self.env_id0, auto_reset=int(self.auto_reset),
                                 stop_on_bounds=int(self.stopOnBoundsExceeded), apply_noise=int(self.applyNoise), device=self.device.index)
        h = _lib.Handle(self.PREFIX, C.byref(p), C.byref(cfg))
        f = self.flow
        nt, ny, nx, _ = f.shape
        _lib.check(h.lib.mvrl_auv_set_flow(h._h, _lib.ptr(f._uv), nt, ny, nx, 2, f.dx, f.dy, f.dt))
        return h

    # -- views ---------------------------------------------------------------
    @property
    def position(self):
        return self._state[0:2, :self.num_envs].T

    @property
    def heading(self):
        return self._state[2, :self.num_envs]

    @property
    def velocities(self):
        return self._state[3:6, :self.num_envs].T

    @property
    def headingTarget(self):
        return self._target[0, :self.num_envs]

    @property
    def flowDataTimeOffset(self):
        return self._target[1, :self.num_envs]

    def reset(self, applyNoise=None, fixedInitialValues=None, mask=None):
        """verySimpleAuv.py:216-262.  ``fixedInitialValues`` = (position ``[N, 2]`` or
        ``[2]``, heading, headingTarget) as in the reference; the draws come from
        Philox keyed on (seed, global env id, episode) instead of the global numpy RNG."""
        h = self._get_handle()
        noise = self.applyNoise if applyNoise is None else bool(applyNoise)
        if noise != self.applyNoise:   # a per-call switch upstream: flip it for this reset only, no new handle
            _lib.check(h.lib.mvrl_auv_set_apply_noise(h._h, int(noise)))
        m = self._begin_reset(mask)
        init = None
        if fixedInitialValues is not None:
            pos, heading, target = fixedInitialValues
            n = self.num_envs
            init = torch.zeros((4, self.ld), dtype=self.dtype, device=self.device)
            p = torch.as_tensor(pos, dtype=self.dtype, device=self.device).reshape(-1, 2)
            init[0:2, :n] = (p.expand(n, 2) if p.shape[0] == 1 else p).T
            init[2, :n] = torch.as_tensor(heading, dtype=self.dtype, device=self.device)
            init[3, :n] = torch.as_tensor(target, dtype=self.dtype, device=self.device)
        _lib.check(h.lib.mvrl_auv_reset(h._h, self.num_envs, self.ld, C.byref(self._bufs), _lib.ptr(m), _lib.ptr(init),
                                        _lib.current_stream(self.device)))
        if noise != self.applyNoise:   # the step kernel's auto-resets keep the constructor's setting
            _lib.check(h.lib.mvrl_auv_set_apply_noise(h._h, int(self.applyNoise)))
        return self.state


def cyl_waypoints(Rcyl=1.33, xCyl=(2.5, 0.)):
    """verySimpleAuv_cyl.py:29-41: 21 way-points (x, y, target heading) on an arc around the cylinder and the
    radius inside which a way-point counts as reached.  Host set-up, exactly the reference's numpy expressions."""
    Rwp = Rcyl * 1.3
    t = np.linspace(-30, 30, 21) * np.pi / 180.
    return np.vstack([-Rwp * np.cos(t) + xCyl[0], Rwp * np.sin(t) + xCyl[1], -t]).T, Rcyl * 0.05


class AuvCylVecEnv(AuvVecEnv):
    """N legacy ``AuvEnvCyl`` environments (verySimpleAuv_cyl.py:22-345): the position / heading targets walk
    along the way-point list, V0 observation scaling, bounds +-2, 1200-step episodes.  ``fixedInitialValues``
    = (position, heading[, ignored]).  The way-point index of an environment survives resets, as upstream."""
    VARIANT = _lib.AUV_CYL
    BOUNDS = 2.

    def __init__(self, num_envs, flow, maxSteps=1200, **kw):
        super().__init__(num_envs, flow, maxSteps=maxSteps, **kw)
        self.Rcyl, self.xCyl = 1.33, np.array([2.5, 0.])
        self.waypoints, self.wpThreshold = cyl_waypoints(self.Rcyl, self.xCyl)

    @property
    def iWp(self):
        return self._iwp[:self.num_envs]

    @property
    def positionTarget(self):
        wp = torch.as_tensor(self.waypoints[:, :2], dtype=self.dtype, device=self.device)
        return wp[self.iWp.long()]

    def reset(self, applyNoise=None, fixedInitialValues=None, mask=None):
        if fixedInitialValues is not None:
            pos, heading = fixedInitialValues[0], fixedInitialValues[1]
            fixedInitialValues = (pos, heading, 0.)
        return super().reset(applyNoise=applyNoise, fixedInitialValues=fixedInitialValues, mask=mask)
