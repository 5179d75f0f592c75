"""Batched BlueROV2 Heavy 3DoF engine (kernel K3): host-side constants with the
reference's attribute names (dynamicsModel_BlueROV2_Heavy_3DoF.py:39-112) and
the vectorised env (…_3DoF.py:375-514).  All numerics run in libmvrl."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import ACT_RPM, ACT_SETPOINT
from ._envbase import _Versioned
from .rov6 import _RovDerivs, _RovHandle, _RovVecEnv


class Rov3Constants(_Versioned):
    def __init__(self):
        self.rho_f = 1000.
        self.m = 11.4
        self.dispVol = self.m / self.rho_f
        self.Length = 0.457
        self.Width = 0.338
        self.CB = np.zeros(3)
        self.CG = np.array([0., 0., 0.02])
        self.I = np.array([[0.16, 0., 0.], [0., 0.16, 0.], [0., 0., 0.16]])
        self.Xudot, self.Yvdot, self.Nrdot = -5.5, -12.7, -0.12
        self.Yrdot = self.Nvdot = 0.
        self.Xuu, self.Yvv, self.Nrr = -18.18, -21.66, -1.55
        self.Yrr = self.Ypp = self.Nvv = self.Npp = 0.
        self.Xu, self.Yv, self.Nr = -4.03, -6.22, -0.07
        self.Yr = self.Yp = self.Nv = self.Np = 0.
        self.D_thruster = 0.1
        self.alphaThruster = 45. / 180. * np.pi
        self.l_x, self.l_y = 0.156, 0.111
        self.Kt_thruster = 40. / (1000. * (3500. / 60.) ** 2. * self.D_thruster ** 4.)
        # allocation with Length/2 arms, 3DoF.py:104-112
        A = np.array([[1., 1., -1., -1.], [1., -1., 1., -1.], [1., 1., 1., 1.]])
        A[0, :] = A[0, :] * np.cos(self.alphaThruster)
        A[1, :] = A[1, :] * np.sin(self.alphaThruster)
        A[2, :] = A[2, :] * np.sin(self.alphaThruster) * self.Length / 2.
        self.A = A
        self.Ainv = np.linalg.pinv(A)
        self.rpmMax, self.rpmDeadband = 3500., 300.
        self.pid = {"windup": np.array([2., 2., 90. / 180. * np.pi]), "Kp": np.array([20., 20., 20.]),
                    "Ki": np.array([0.1, 0.1, 0.1]), "Kd": np.array([5., 5., 0.5]), "max": np.array([150., 150., 100.])}

    def massMatrix(self):
        """3DoF.py:198-206."""
        m, xg, yg = self.m, self.CG[0], self.CG[1]
        Mrb = np.array([[m, 0., -m * yg], [0., m, m * xg], [-m * yg, m * xg, self.I[2, 2]]])
        return Mrb + -1. * np.diag([self.Xudot, self.Yvdot, self.Nrdot])

    def to_struct(self):
        p = _lib.MvrlRov3Params()
        for name in ("rho_f", "m", "Length", "dispVol", "Xudot", "Yvdot", "Nrdot", "Xu", "Yv", "Yr", "Nv", "Nr",
                     "Xuu", "Yvv", "Yrr", "Nvv", "Nrr", "D_thruster", "alphaThruster", "l_x", "l_y"):
            setattr(p, name, float(getattr(self, name)))
        p.xg, p.yg, p.Izz = float(self.CG[0]), float(self.CG[1]), float(self.I[2, 2])
        p.thrust_coef = self.rho_f * self.D_thruster ** 4. * self.Kt_thruster
        p.rpm_max, p.rpm_deadband = self.rpmMax, self.rpmDeadband
        M = self.massMatrix()
        p.M[:] = list(M.reshape(-1))
        p.Minv[:] = list(np.linalg.inv(M).reshape(-1))
        p.Ainv[:] = list(np.asarray(self.Ainv, dtype=float).reshape(-1))
        p.pid_Kp[:] = list(self.pid["Kp"]); p.pid_Ki[:] = list(self.pid["Ki"]); p.pid_Kd[:] = list(self.pid["Kd"])
        p.pid_windup[:] = list(self.pid["windup"]); p.pid_max[:] = list(self.pid["max"])
        return p


class Rov3Handle(_RovHandle):
    PREFIX = "mvrl_rov3"


class BlueROV2Heavy3DoFVecEnv(_RovVecEnv):
    """Batched ``BlueROV2Heavy3DoFEnv`` (3DoF.py:375-514): 6 states, 5
    observations; "setpoint" actions (3 in [-1, 1], reference semantics) or
    "rpm" (4 thruster rpm FP AP FS AS, stateless)."""
    HANDLE, CONSTANTS = Rov3Handle, Rov3Constants
    STATE_DIM, OBS_DIM, SP_DIM, PATH_DIM, CTRL_DIM, AUX_DIM = 6, 5, 3, 4, 7, 7
    ACTION_DIM = {ACT_RPM: 4, ACT_SETPOINT: 3}
    HISTORY_COLUMNS = (["t"] + ["x%d" % i for i in range(6)] + ["F%d" % i for i in range(3)] + ["u%d" % i for i in range(4)]
                       + ["x_d", "y_d", "psi_d"])  # 3DoF.py:503-508


class Rov3Derivs(_RovDerivs):
    """Batched ``BlueROV2Heavy3DoF.derivs`` (3DoF.py:128-296) through
    ``mvrl_rov3_derivs``.  state [6, N]; rpm mode: act [4, N]; set-point mode:
    t [N], setpoint [3, N], ctrl [7, N] (updated in place)."""
    HANDLE, CONSTANTS, CTRL_ROWS, AUX_ROWS = Rov3Handle, Rov3Constants, 7, 7

    def __init__(self, consts=None, dtype=torch.float64, action_mode="setpoint", device="cuda"):
        super().__init__(consts, dtype, action_mode, device)

    def thrusterModel(self, u, rpm):
        """(Fthruster, Xthruster), 3DoF.py:114-126; u, rpm: tensors [N]."""
        h = self._get_handle()
        u = u.to(device=self.device, dtype=self.dtype).contiguous()
        rpm = rpm.to(device=self.device, dtype=self.dtype).contiguous()
        F, X = torch.empty_like(u), torch.empty_like(u)
        _lib.check(h.fn("thruster_model")(h._h, u.numel(), _lib.ptr(u), _lib.ptr(rpm), _lib.ptr(F), _lib.ptr(X),
                                          _lib.current_stream(self.device)))
        return F, X
