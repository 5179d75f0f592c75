"""Drop-in for the reference module ``dynamicsModel_BlueROV2_Heavy_6DoF``:
``BlueROV2Heavy6DoF_PID_controller``, ``BlueROV2Heavy6DoF`` and
``BlueROV2Heavy6DoFEnv`` with the reference's constructor signatures,
attributes and return conventions (one vehicle, numpy in / numpy out, old-Gym
4-tuple), plus ``BlueROV2Heavy6DoFVecEnv`` for batches.

Every number is produced by the CUDA kernels of libmvrl (fp64, one
environment); this file only marshals.  Differences from the reference, all
deliberate: ``env.step`` integrates with fixed-step RK4 x ``nSub`` instead of
scipy's adaptive RK45 (BASELINE.json north star), and ``reset()`` without a
set-point draws the path instead of raising (6DoF.py:497 is broken upstream).
The plotting helpers of the reference module are out of scope.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib, resources
from ._envbase import _RovEnv
from .rov6 import BlueROV2Heavy6DoFVecEnv, Rov6Constants, Rov6Derivs, Rov6Handle  # noqa: F401

_F64 = torch.float64


def _col(values, device):
    """numpy vector -> [k, 1] fp64 CUDA tensor (one environment, SoA)."""
    return torch.as_tensor(np.asarray(values, dtype=np.float64).reshape(-1, 1), device=device)


class BlueROV2Heavy6DoF_PID_controller(object):
    """6DoF.py:27-73.  State (eOld, eInt, tOld) lives on the host like the
    reference's; ``computeControlForces`` runs ``mvrl_rov6_pid``."""

    def __init__(self, setPoint, device="cuda"):
        self.setPoint = setPoint
        self._device = device
        self._handle = None
        self._consts = Rov6Constants()
        self.reset()

    def reset(self):
        self.eOld = None
        self.eInt = np.zeros(6)
        self.tOld = 0.

    def computeControlForces(self, x, y, z, phi, theta, psi, t):
        if self._handle is None:
            self._handle = Rov6Handle(self._consts, _F64, "setpoint", device=torch.device(self._device).index or 0)
        dev = torch.device("cuda", self._handle.cfg.device)
        ctrl = np.zeros(13)
        ctrl[0:6] = np.nan if self.eOld is None else self.eOld
        ctrl[6:12] = self.eInt
        ctrl[12] = self.tOld
        d_ctrl = _col(ctrl, dev)
        out = torch.empty((6, 1), dtype=_F64, device=dev)
        h = self._handle
        # named tensors: a temporary would be freed (and its block reused by the next one) before the kernel reads it
        d_pose, d_t, d_sp = _col([x, y, z, phi, theta, psi], dev), _col([t], dev), _col(self.setPoint, dev)
        _lib.check(h.lib.mvrl_rov6_pid(h._h, 1, 1, _lib.ptr(d_pose), _lib.ptr(d_t), _lib.ptr(d_sp), _lib.ptr(d_ctrl), _lib.ptr(out),
                                       _lib.current_stream(dev)))
        c = d_ctrl[:, 0].cpu().numpy()
        self.eOld, self.eInt, self.tOld = c[0:6].copy(), c[6:12].copy(), float(c[12])
        return out[:, 0].cpu().numpy()


class BlueROV2Heavy6DoF(Rov6Constants):
    """6DoF.py:75-442 for one vehicle.  ``controller`` is any object with
    ``computeControlForces(x, y, z, phi, theta, psi, t) -> (6,)``,
    ``.setPoint`` and ``.reset()`` (the reference's injection seam)."""

    def __init__(self, controller, disableThrusters=False, device="cuda"):
        super().__init__()
        self.controller = controller
        self.disableThrusters = disableThrusters
        self.generalisedControlForces = np.zeros(6)
        self.controlVector = np.zeros(8)
        self.rotation_angles = np.zeros(3)
        self.iHat, self.jHat, self.kHat = np.eye(3)
        object.__setattr__(self, "_dev", torch.device(device))
        object.__setattr__(self, "_f_rpm", None)
        object.__setattr__(self, "_f_force", None)

    # lazily built fp64 derivative evaluators (rpm / force modes) sharing these constants
    def _eval(self, mode):
        name = "_f_" + mode
        if getattr(self, name) is None:
            object.__setattr__(self, name, Rov6Derivs(consts=self, dtype=_F64, action_mode=mode, device=self._dev))
        return getattr(self, name)

    def allocateThrust(self):
        """6DoF.py:220-231: rpm demand for ``self.generalisedControlForces`` at the current orientation."""
        f = self._eval("force")
        state = np.zeros(12)
        state[3:6] = self.rotation_angles
        _, aux = f(_col(state, f.device), _col(self.generalisedControlForces, f.device), want_aux=True)
        self.controlVector = aux[12:20, 0].cpu().numpy()
        return self.controlVector

    def thrusterModel(self, rpm):
        """6DoF.py:233-236."""
        f = self._eval("rpm")
        h = f._get_handle()
        r = torch.as_tensor(np.atleast_1d(np.asarray(rpm, dtype=np.float64)), device=f.device).contiguous()
        F = torch.empty_like(r)
        _lib.check(h.lib.mvrl_rov6_thruster_model(h._h, r.numel(), _lib.ptr(r), _lib.ptr(F), _lib.current_stream(f.device)))
        F = F.cpu().numpy()
        return float(F[0]) if np.ndim(rpm) == 0 else F.reshape(np.shape(rpm))

    def updateMovingCoordSystem(self, rotation_angles):
        """6DoF.py:238-242: vehicle axes for intrinsic-XYZ roll/pitch/yaw."""
        self.rotation_angles = np.asarray(rotation_angles, dtype=float)
        dev = self._eval("rpm").device
        out = torch.empty((9, 1), dtype=_F64, device=dev)
        d_ang = _col(self.rotation_angles, dev)
        _lib.check(_lib.load().mvrl_body_axes(_lib.F64, 1, 1, _lib.ptr(d_ang), _lib.ptr(out), _lib.current_stream(dev)))
        self.iHat, self.jHat, self.kHat = out[:, 0].cpu().numpy().reshape(3, 3)

    def _rotate(self, vec, to_vehicle):
        dev = self._eval("rpm").device
        axes = _col(np.concatenate([self.iHat, self.jHat, self.kHat]), dev)
        out = torch.empty((3, 1), dtype=_F64, device=dev)
        d_vec = _col(vec, dev)
        _lib.check(_lib.load().mvrl_frame_rotate(_lib.F64, 1, 1, _lib.ptr(axes), _lib.ptr(d_vec), _lib.ptr(out), int(to_vehicle),
                                                 _lib.current_stream(dev)))
        return out[:, 0].cpu().numpy()

    def globalToVehicle(self, vecGlobal):
        return self._rotate(vecGlobal, True)

    def vehicleToGlobal(self, vecVehicle):
        return self._rotate(vecVehicle, False)

    def forceModel(self, pos, angles, vel, rpms, retComp=False):
        """6DoF.py:253-404 -> (M, RHS), or the 6x5 component matrix if ``retComp``."""
        f = self._eval("rpm")
        state = np.concatenate([np.asarray(pos, float), np.asarray(angles, float), np.asarray(vel, float)])
        _, aux = f(_col(state, f.device), _col(rpms, f.device), want_aux=True)
        aux = aux[:, 0].cpu().numpy()
        if retComp:
            return aux[20:50].reshape(5, 6).T
        return self.massMatrix(), aux[0:6]

    def derivs(self, t, state):
        """6DoF.py:406-442."""
        x, y, z, phi, theta, psi = (float(v) for v in state[:6])
        self.updateMovingCoordSystem(np.array([phi, theta, psi]))
        self.generalisedControlForces = np.asarray(self.controller.computeControlForces(x, y, z, phi, theta, psi, t), dtype=float)
        f = self._eval("force")
        d, aux = f(_col(state, f.device), _col(self.generalisedControlForces, f.device), want_aux=True)
        self.controlVector = aux[12:20, 0].cpu().numpy()
        return d[:, 0].cpu().numpy()


HISTORY_COLUMNS = BlueROV2Heavy6DoFVecEnv.HISTORY_COLUMNS


class BlueROV2Heavy6DoFEnv(_RovEnv):
    """6DoF.py:445-594 for one vehicle (old-Gym API: ``reset() -> obs``,
    ``step() -> (obs, reward, done, {})``).  ``nSub`` = RK4 sub-steps per
    ``dt`` (the reference integrates with adaptive RK45)."""
    _VEC = BlueROV2Heavy6DoFVecEnv

    def _new_vehicle(self, sp):
        self.targetOrientation = sp[3:].copy()
        self.vehicle = BlueROV2Heavy6DoF(BlueROV2Heavy6DoF_PID_controller(sp, device=self._device), device=self._device)

    def _sync_from_device(self):
        v = self._vec
        self.systemState = v.systemState[0].cpu().numpy()
        self.state = v.state[0].cpu().numpy()
        self.path = v.path[0].cpu().numpy()
        sp = v.setPoint[0].cpu().numpy()
        self.vehicle.controller.setPoint = sp
        aux = v._aux[:, 0].cpu().numpy()
        self.vehicle.generalisedControlForces = aux[:6]
        self.vehicle.controlVector = aux[6:]
        c = v._ctrl[:, 0].cpu().numpy()
        ctl = self.vehicle.controller
        ctl.eOld, ctl.eInt, ctl.tOld = (None if np.isnan(c[0]) else c[0:6].copy()), c[6:12].copy(), float(c[12])
        return sp
