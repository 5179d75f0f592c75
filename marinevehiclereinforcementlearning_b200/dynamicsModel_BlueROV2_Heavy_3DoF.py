"""Drop-in for the reference module ``dynamicsModel_BlueROV2_Heavy_3DoF``:
``BlueROV2Heavy3DoF`` and ``BlueROV2Heavy3DoFEnv`` with the reference's
constructor signatures, attributes and return conventions (one vehicle, numpy
in / numpy out, old-Gym 4-tuple), plus ``BlueROV2Heavy3DoFVecEnv`` for batches.

Every number is produced by the CUDA kernels of libmvrl (fp64, one
environment); this file only marshals.  As for the 6DoF module, ``env.step``
integrates with fixed-step RK4 x ``nSub`` instead of scipy's adaptive RK45.
``lineOfSight`` / ``LOSNavigation`` (3DoF.py:517-607) run as the ``mvrl_los_navigation`` kernel; the plotting
helpers of the reference module are out of scope (SURVEY.md section 2, row 10).
"""
import numpy as np
import torch

from . import _lib, resources  # noqa: F401
from ._envbase import _RovEnv
from .resources import angleError  # noqa: F401  (the reference module re-exports it)
from .rov3 import BlueROV2Heavy3DoFVecEnv, Rov3Constants, Rov3Derivs, Rov3Handle  # noqa: F401

_F64 = torch.float64


def _col(values, device):
    return torch.as_tensor(np.asarray(values, dtype=np.float64).reshape(-1, 1), device=device)


class BlueROV2Heavy3DoF(Rov3Constants):
    """3DoF.py:25-296 for one vehicle.  The built-in PID state (``eOld``,
    ``eInt``, ``tOld``) lives on the host like the reference's and is mutated
    by every ``derivs`` call."""

    def __init__(self, setPoint, device="cuda"):
        super().__init__()
        self.setPoint = setPoint
        self.eOld = None
        self.eInt = np.zeros(3)
        self.tOld = 0.
        self.generalisedControlForces = np.zeros(3)
        self.controlVector = np.zeros(4)
        object.__setattr__(self, "_dev", torch.device(device))
        object.__setattr__(self, "_f", None)

    def __setattr__(self, name, value):
        # controller state / outputs are not vehicle constants: no handle rebuild
        if name in ("setPoint", "eOld", "eInt", "tOld", "generalisedControlForces", "controlVector"):
            object.__setattr__(self, name, value)
        else:
            super().__setattr__(name, value)

    def _eval(self):
        if self._f is None:
            object.__setattr__(self, "_f", Rov3Derivs(consts=self, dtype=_F64, action_mode="setpoint", device=self._dev))
        return self._f

    def thrusterModel(self, u, v, rpm):
        """3DoF.py:114-126 -> (Fthruster, Xthruster)."""
        f = self._eval()
        shape = np.broadcast(np.asarray(u), np.asarray(rpm)).shape
        uu = torch.as_tensor(np.broadcast_to(np.asarray(u, dtype=np.float64), shape).reshape(-1).copy(), device=f.device)
        rr = torch.as_tensor(np.broadcast_to(np.asarray(rpm, dtype=np.float64), shape).reshape(-1).copy(), device=f.device)
        F, X = f.thrusterModel(uu, rr)
        F, X = F.cpu().numpy().reshape(shape), X.cpu().numpy().reshape(shape)
        return (float(F), float(X)) if shape == () else (F, X)

    def derivs(self, t, state):
        """3DoF.py:128-296."""
        f = self._eval()
        ctrl = np.zeros(7)
        ctrl[0:3] = np.nan if self.eOld is None else self.eOld
        ctrl[3:6] = self.eInt
        ctrl[6] = self.tOld
        d_ctrl = _col(ctrl, f.device)
        d, aux = f(_col(state, f.device), t=_col([t], f.device).reshape(1), setpoint=_col(self.setPoint, f.device), ctrl=d_ctrl, want_aux=True)
        c = d_ctrl[:, 0].cpu().numpy()
        self.eOld, self.eInt, self.tOld = c[0:3].copy(), c[3:6].copy(), float(c[6])
        aux = aux[:, 0].cpu().numpy()
        self.generalisedControlForces = aux[0:3].copy()
        self.controlVector = aux[3:7].copy()
        return d[:, 0].cpu().numpy()


HISTORY_COLUMNS = BlueROV2Heavy3DoFVecEnv.HISTORY_COLUMNS


class BlueROV2Heavy3DoFEnv(_RovEnv):
    """3DoF.py:375-514 for one vehicle (old-Gym API).  ``nSub`` = RK4 sub-steps per ``dt``."""
    _VEC = BlueROV2Heavy3DoFVecEnv

    def _new_vehicle(self, sp):
        self.targetHeading = float(sp[2])
        self.vehicle = BlueROV2Heavy3DoF(sp, device=self._device)

    def _sync_from_device(self):
        v = self._vec
        self.systemState = v.systemState[0].cpu().numpy()
        self.state = v.state[0].cpu().numpy()
        self.path = v.path[0].cpu().numpy()
        veh = self.vehicle
        veh.setPoint = v.setPoint[0].cpu().numpy()
        aux = v._aux[:, 0].cpu().numpy()
        veh.generalisedControlForces, veh.controlVector = aux[:3], aux[3:]
        c = v._ctrl[:, 0].cpu().numpy()
        veh.eOld, veh.eInt, veh.tOld = (None if np.isnan(c[0]) else c[0:3].copy()), c[3:6].copy(), float(c[6])
        return veh.setPoint


def _los_actions(obs_fm, rnav):
    """[5, N] CUDA tensor -> [3, N] actions through ``mvrl_los_navigation``."""
    n = obs_fm.shape[1]
    act = torch.empty((3, n), dtype=obs_fm.dtype, device=obs_fm.device)
    _lib.check(_lib.load().mvrl_los_navigation(_lib.torch_dtype_code(obs_fm.dtype), n, n, _lib.ptr(obs_fm), _lib.ptr(act), float(rnav),
                                               _lib.current_stream(obs_fm.device)))
    return act


def lineOfSight(p0, p1, Rnav):
    """3DoF.py:517-583: target point on the path segment p0 -> p1 (relative to the vehicle) within the
    line-of-sight radius.  numpy 2-vectors in, numpy 2-vector out."""
    _lib.require_cuda()
    obs = torch.as_tensor(np.concatenate([np.asarray(p0, float), np.asarray(p1, float), [0.]]).reshape(5, 1), device="cuda")
    return _los_actions(obs, Rnav)[:2, 0].cpu().numpy()


class LOSNavigation(object):
    """3DoF.py:586-607: SB3-like ``predict(obs, deterministic)`` -> (actions, states).  One observation
    ``(5,)`` (numpy, like the reference) or a batch: numpy / torch ``[N, 5]`` -> ``[N, 3]`` (torch stays on the device)."""
    Rnav = 0.5

    def __init__(self):
        pass

    def predict(self, obs, deterministic=True):
        states = obs
        _lib.require_cuda()
        if isinstance(obs, torch.Tensor):
            o = obs if obs.is_cuda else obs.cuda()
            single = o.dim() == 1
            fm = o.reshape(-1, 5).T.contiguous()
            act = _los_actions(fm, self.Rnav).T
            return (act[0] if single else act), states
        o = np.asarray(obs, dtype=np.float64)
        fm = torch.as_tensor(np.ascontiguousarray(o.reshape(-1, 5).T), device="cuda")
        act = _los_actions(fm, self.Rnav).T.cpu().numpy()
        return (act[0] if o.ndim == 1 else act), states
