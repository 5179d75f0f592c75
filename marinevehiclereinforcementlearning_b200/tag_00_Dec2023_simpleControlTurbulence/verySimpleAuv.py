"""Drop-in for tag_00_Dec2023_simpleControlTurbulence/verySimpleAuv.py:
``AuvEnv`` (one vehicle, numpy in / numpy out, old-Gym 4-tuple), ``PDController``
and ``make_env``, plus ``AuvVecEnv`` for batches.  The env step runs in the
``auv_step`` CUDA kernel (fp64 for the single-vehicle class)."""
import numpy as np
import torch

from .._gymshim import Box, Env
from ..auv import AUX_COLUMNS, AuvVecEnv  # noqa: F401
from . import flowGenerator
from .resources import headingError  # noqa: F401


class PDController(object):
    """verySimpleAuv.py:22-50: PD law on ``obs[:3]`` with an SB3-like ``predict``.
    Works on one observation ``(obs_dim,)`` (numpy, like the reference) or on a
    batch ``[N, obs_dim]`` of numpy arrays / torch tensors (stays on the device)."""

    def __init__(self, dt, P=[1., 1., 1.], D=[0.05, 0.05, 0.01], noiseSigma=None):
        self.P = np.array(P)
        self.D = np.array(D)
        self.dt = dt
        self.oldObs = None
        self.noiseSigma = noiseSigma

    def predict(self, obs, deterministic=True):
        states = obs
        if isinstance(obs, torch.Tensor):
            x = obs[..., :3]
            P = torch.as_tensor(self.P, dtype=x.dtype, device=x.device)
            D = torch.as_tensor(self.D, dtype=x.dtype, device=x.device)
            if self.oldObs is None:
                self.oldObs = x.clone()
            actions = torch.clamp(x * P + (x - self.oldObs) / self.dt * D, -1., 1.)
            if self.noiseSigma is not None:
                actions = actions + torch.randn_like(actions) * self.noiseSigma
            self.oldObs = x.clone()
            return torch.clamp(actions, -1., 1.), states
        x = np.asarray(obs)[..., :3]
        if self.oldObs is None:
            self.oldObs = x
        actions = np.clip(x * self.P + (x - self.oldObs) / self.dt * self.D, -1., 1.)
        if self.noiseSigma is not None:
            actions += np.random.normal(loc=0., scale=self.noiseSigma, size=actions.shape)
        self.oldObs = x
        return np.clip(actions, -1., 1.), states


# column order of one timeHistory row, verySimpleAuv.py:389-401
HISTORY_COLUMNS = AuvVecEnv.HISTORY_COLUMNS


class AuvEnv(Env):
    """verySimpleAuv.py:76-416 for one vehicle.  ``flow`` may be passed explicitly
    (a ``flowGenerator.ReconstructedFlow`` on the same device, fp64); otherwise
    ``./turbulenceData`` is loaded like the reference does."""

    def __init__(self, seed=None, dt=0.02, noiseMagCoeffs=0.0, noiseMagActuation=0.0,
                 currentVelScale=1.0, currentTurbScale=2.0, stopOnBoundsExceeded=True, flow=None, device="cuda"):
        super(AuvEnv, self).__init__()
        self.seed = seed
        self._max_episode_steps = 250
        self.stopOnBoundsExceeded = stopOnBoundsExceeded
        self.iStep = 0
        self.dt = dt
        self.state = None
        self.steps_beyond_done = None
        self.perr_0 = np.zeros(2)
        self.herr_o = 0.
        if flow is None:
            flow = flowGenerator.ReconstructedFlow("./turbulenceData", dtype=torch.float64, device=device)
        self.flow = flow
        self.flow.scale(11., currentVelScale, currentTurbScale, translate=(-1.65, -1.1))  # verySimpleAuv.py:104
        self.timeHistory = []
        self.xMinMax = [-1, 1]
        self.yMinMax = [-1, 1]
        self.m, self.Izz = 11.4, 0.16
        self.Xuu, self.Yvv, self.Nrr = -18.18 * 2.21, -21.66 * 4.87, -1.55
        self.Xu, self.Yv, self.Nr = -4.03 * 2.21, -6.22 * 4.87, -0.07
        self.maxForce, self.maxMoment = 150., 20.
        self.noiseMagCoeffs = noiseMagCoeffs
        self.noiseMagActuation = noiseMagActuation
        self.lenAction = 3
        self.action_space = Box(low=-1.0, high=1.0, shape=(self.lenAction,), dtype=np.float32)
        lenState = 9 + 2
        self.observation_space = Box(-1 * np.ones(lenState, dtype=np.float32), np.ones(lenState, dtype=np.float32), shape=(lenState,))
        self._vec = None

    _COEFFS = ("m", "Izz", "Xuu", "Yvv", "Nrr", "Xu", "Yv", "Nr", "maxForce", "maxMoment", "noiseMagCoeffs", "noiseMagActuation",
               "stopOnBoundsExceeded", "_max_episode_steps", "dt")

    _VEC = AuvVecEnv

    def _engine(self):
        if self._vec is None:
            self._vec = self._VEC(1, self.flow, seed=0 if self.seed is None else int(self.seed), dt=self.dt, dtype=self.flow.dtype,
                                  auto_reset=False, record_aux=True, record_terminal_obs=False)
        v = self._vec
        for name in self._COEFFS:  # attributes edited on the env (as reference users do) reach the kernel
            setattr(v, name, getattr(self, name))
        v.xMinMax, v.yMinMax = [float(x) for x in self.xMinMax], [float(x) for x in self.yMinMax]
        return v

    def _sync(self):
        v = self._vec
        s = v._state[:, 0].cpu().numpy()
        self.position, self.heading, self.velocities = s[0:2].copy(), float(s[2]), s[3:6].copy()
        self.state = v.state[0].cpu().numpy()
        e = v._err_o[:, 0].cpu().numpy()
        self.perr_o, self.herr_o = e[0:2].copy(), float(e[2])

    def dataToState(self, pos, heading, velocities):
        """verySimpleAuv.py:147-214 (V3) for the given pose, against the stored previous errors."""
        perr = self.positionTarget - np.asarray(pos, dtype=float)
        herr = headingError(self.headingTarget, heading)
        herr_o, perr_o = (herr, perr) if self.herr_o is None else (self.herr_o, self.perr_o)
        c = lambda x: min(1., max(-1., x))
        return np.concatenate([[c(perr[0]), c(perr[1]), c(herr / (45. / 180. * np.pi)), c(herr - herr_o),
                                c(perr[0] - perr_o[0]), c(perr[1] - perr_o[1])], np.clip(velocities, -1., 1.), np.zeros(2)])

    def reset(self, keepTimeHistory=False, applyNoise=True, fixedInitialValues=None):
        v = self._engine()
        v.reset(applyNoise=applyNoise, fixedInitialValues=fixedInitialValues)
        m = v._mults[:, 0].cpu().numpy()
        (self.mMult, self.IMult, self.XuuMult, self.YvvMult, self.NrrMult, self.XuMult, self.YvMult, self.NrMult,
         self.XactMult, self.YactMult, self.NactMult) = (float(x) for x in m)
        self.positionTarget = np.zeros(2)
        self.headingTarget = float(v.headingTarget[0])
        self.flowDataTimeOffset = float(v.flowDataTimeOffset[0])
        self.time = 0
        self.iStep = 0
        self.steps_beyond_done = 0
        self.timeHistory = []
        self._sync()
        self.positionStart = self.position.copy()
        self.headingStart = self.heading
        return self.state

    def step(self, action):
        self.iStep += 1
        self.time += self.dt
        action = np.asarray(action, dtype=np.float64)
        v = self._engine()
        a = torch.as_tensor(action.reshape(1, 3), device=v.device)
        _, rew, done, _ = v.step(a)
        reward, done = float(rew[0]), bool(done[0])
        self._sync()
        aux = v._aux[:, 0].cpu().numpy()
        row = np.concatenate([[self.iStep, self.time, reward], self.position, [self.heading], self.positionTarget, [self.headingTarget],
                              aux[0:6], self.velocities, aux[6:9], aux[9:14], action, self.state])
        self.timeHistory.append(dict(zip(HISTORY_COLUMNS, row)))
        if done:
            import pandas
            self.timeHistory = pandas.DataFrame(self.timeHistory)
            self.steps_beyond_done += 1
        else:
            self.steps_beyond_done = 0
        return self.state, reward, done, {}


def make_env(rank, seed=0, env_kwargs={}):
    """verySimpleAuv.py:419-433: thunk factory for (Subproc)VecEnv-style constructors."""
    def _init():
        return AuvEnv(seed=seed + rank, **env_kwargs)
    return _init
