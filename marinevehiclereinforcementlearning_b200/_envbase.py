"""Host plumbing shared by the batched envs (rov6.py, rov3.py, auv.py) and the derivative evaluators: the cached
library handle, version tracking of vehicle constants, the batched env body - device buffers, views, reset / step,
episode statistics and checkpoints - and the single-vehicle ROV env of the drop-in modules."""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._gymshim import Box, Env


class _HandleCache:
    """Keeps the handle ``_new_handle()`` built for the last key; a new key (a changed constant or flag) rebuilds it."""
    _handle = _handle_key = None

    def _cached_handle(self, key):
        if key != self._handle_key:
            self._handle, self._handle_key = self._new_handle(), key
        return self._handle


class _Versioned:
    """Vehicle constants whose handles are rebuilt when an attribute is assigned: ``fingerprint()`` changes with every
    assignment (and with ``touch()``)."""

    def __setattr__(self, name, value):
        object.__setattr__(self, name, value)
        object.__setattr__(self, "_version", getattr(self, "_version", 0) + 1)

    def touch(self):
        """Call after modifying an array attribute in place (e.g. ``rov.CG[2] = 0.1``)
        so that handles built from these constants are refreshed."""
        object.__setattr__(self, "_version", self._version + 1)

    def fingerprint(self):
        return (id(self), self._version)


class _VecEnv(_HandleCache):
    """N environments stepped by one fused CUDA kernel, the batch following the SB3 ``VecEnv`` convention (``step`` ->
    obs, rewards, dones, infos; auto-reset with ``terminal_observation``).  Tensors stay on the device.  Every array is
    structure-of-arrays ``[field, ld]``; ``obs`` / ``actions`` are exposed as ``[N, k]`` views of them (``*_fm`` gives
    the feature-major tensors for transposition-free policies).

    A subclass sets ``lenAction`` before calling ``__init__`` with the prefix of its C entries (``<prefix>_step`` among
    them) and declares:
    * ``STATE_DIM``, ``OBS_DIM``, ``AUX_DIM``: rows of the state, observation and aux (log) buffers;
    * ``BUFFERS``: the ctypes struct of buffer pointers its C entries take, field ``f`` filled from attribute ``_f``
      (``ep_stats`` from ``_stats``), and ``_extra_buffers()``, which allocates the buffers of its own fields;
    * ``_get_handle()``: its handle key through ``_cached_handle``, and ``_new_handle()``, the ``_lib.Handle``;
    * ``_STATE_KEYS``: what ``state_dict()`` keeps, device tensors or host flags;
    * ``HISTORY_COLUMNS``: the columns of the single-vehicle env's ``timeHistory`` (``vec_tools.TrajectoryRecorder``)."""

    def __init__(self, prefix, num_envs, device, dtype, dt, maxSteps, seed, env_id0, auto_reset, record_aux,
                 record_terminal_obs, collect_stats):
        self.num_envs = int(num_envs)
        self.device, self.dtype = device, dtype
        self.dt, self._max_episode_steps = float(dt), int(maxSteps)
        self.seed, self.env_id0, self.auto_reset = int(seed), int(env_id0), bool(auto_reset)
        self.lenObs = self.OBS_DIM
        self.ld = max(32, ((self.num_envs + 31) // 32) * 32)    # an empty batch still owns (non-null) buffers
        z = self._zeros
        self._state, self._action, self._obs = z(self.STATE_DIM), z(self.lenAction), z(self.OBS_DIM)
        self._reward = z()
        self._done = z(dtype=torch.uint8)
        self._istep = z(dtype=torch.int32)
        self._episode = z(dtype=torch.int32)  # reinterpreted as uint32
        self._terminal_obs = z(self.OBS_DIM) if (record_terminal_obs and auto_reset) else None
        self._aux = z(self.AUX_DIM) if record_aux else None
        self._stats = torch.zeros(8, dtype=torch.float64, device=device) if collect_stats else None
        if self._stats is not None:
            self._reset_stats()
        self._extra_buffers()
        bufs = {f: getattr(self, "_stats" if f == "ep_stats" else "_" + f) for f, _ in self.BUFFERS._fields_}
        self._bufs = self.BUFFERS(**{f: None if t is None else t.data_ptr() for f, t in bufs.items()})
        self._needs_episode_bump = False
        self._step_entry = getattr(_lib.load(), prefix + "_step")   # looked up once: step_async is called eagerly

    def _zeros(self, *rows, dtype=None):
        """A zero device buffer ``[*rows, ld]`` (the env's dtype unless given)."""
        return torch.zeros(rows + (self.ld,), dtype=self.dtype if dtype is None else dtype, device=self.device)

    def _reset_stats(self):
        self._stats.zero_()
        self._stats[3] = float("inf")
        self._stats[4] = float("-inf")

    # -- views -----------------------------------------------------------------
    @property
    def obs_fm(self):
        return self._obs[:, :self.num_envs]

    @property
    def actions_fm(self):
        return self._action[:, :self.num_envs]

    @property
    def state(self):
        return self.obs_fm.T

    @property
    def iStep(self):
        return self._istep[:self.num_envs]

    @property
    def time(self):
        return self._istep[:self.num_envs].to(torch.float64) * self.dt

    # -- reset / step ------------------------------------------------------------
    def _begin_reset(self, mask):
        """Episode counters of the environments a reset restarts (all of them, or where ``mask`` is set) advance, except at
        the first reset; returns ``mask`` as a uint8 device tensor (or None) for the reset entry."""
        if self._needs_episode_bump:
            if mask is None:
                self._episode += 1
            else:
                self._episode[:self.num_envs] += torch.as_tensor(mask).to(device=self.device, dtype=torch.int32)
        self._needs_episode_bump = True
        return None if mask is None else torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()

    def set_actions(self, actions):
        """Copy ``actions`` ([N, A] or feature-major [A, N]) into the SoA action buffer."""
        if actions.data_ptr() == self._action.data_ptr():
            return
        a = actions.to(device=self.device, dtype=self.dtype, non_blocking=True)
        if a.dim() == 2 and a.shape == (self.num_envs, self.lenAction):
            self.actions_fm.copy_(a.T)
        elif a.dim() == 2 and a.shape == (self.lenAction, self.num_envs):
            self.actions_fm.copy_(a)
        else:
            raise ValueError("actions must be [%d, %d] or [%d, %d], got %s" %
                             (self.num_envs, self.lenAction, self.lenAction, self.num_envs, tuple(a.shape)))

    def step_async(self, actions=None):
        """Launch the fused step kernel on the current stream (no sync)."""
        if actions is not None:
            self.set_actions(actions)
        h = self._get_handle()
        _lib.check(self._step_entry(h._h, self.num_envs, self.ld, C.byref(self._bufs), _lib.current_stream(self.device)))

    def step(self, actions=None):
        self.step_async(actions)
        n = self.num_envs
        infos = {}
        if self._terminal_obs is not None:
            infos["terminal_observation"] = self._terminal_obs[:, :n].T
        return self.state, self._reward[:n], self._done[:n].bool(), infos

    # -- episode statistics (K5): device-side accumulators + optional all-reduce
    def episode_stats(self, reduce_group=None, reset=True):
        """{episodes, mean_length, mean_return, min_return, max_return,
        nonfinite}.  When torch.distributed is initialised the 8 accumulators
        are all-reduced over the process group (NCCL on GPUs) - the only
        collective of the framework, off the step path.  Episodes are counted
        where they END INSIDE THE KERNEL, i.e. with ``auto_reset=True``; an env
        created with ``auto_reset=False`` keeps integrating past ``done`` like
        the reference (6DoF.py:589-592) and reports 0 episodes here."""
        if self._stats is None:
            raise RuntimeError("collect_stats=False")
        from .distributed import reduce_episode_stats
        out = reduce_episode_stats(self._stats, group=reduce_group)
        if reset:
            self._reset_stats()
        return out

    # -- checkpoint / resume -------------------------------------------------------
    def state_dict(self):
        d = {}
        for k in self._STATE_KEYS:
            v = getattr(self, k)
            d[k] = v.clone() if torch.is_tensor(v) else v
        return d

    def load_state_dict(self, d):
        for k, v in d.items():
            cur = getattr(self, k)
            if torch.is_tensor(cur):
                cur.copy_(v)
            else:   # a host flag
                setattr(self, k, bool(v))
        self._needs_episode_bump = True


class _RovEnv(Env):
    """One vehicle of a batched ROV env ``_VEC`` with the reference's Gym API (``reset() -> obs``, ``step() -> (obs,
    reward, done, {})``), fp64, its attributes synced from the device after every call.  ``nSub`` = RK4 sub-steps per
    ``dt`` (the reference integrates with adaptive RK45).  A subclass declares ``_new_vehicle(sp)`` (the vehicle object
    and the target attribute of a reset) and ``_sync_from_device()``, which returns the set-point it synced."""

    def __init__(self, seed=None, dt=0.2, maxSteps=250, nSub=8, device="cuda"):
        super().__init__()
        self.seed = seed
        self.dt = dt
        self._max_episode_steps = maxSteps
        self.nSub = nSub
        self.lenAction = self._VEC.ACTION_DIM[_lib.ACT_SETPOINT]
        self.action_space = Box(low=-1.0, high=1.0, shape=(self.lenAction,), dtype=np.float32)
        self.lenObs = self._VEC.OBS_DIM
        self.observation_space = Box(-1 * np.ones(self.lenObs, dtype=np.float32), np.ones(self.lenObs, dtype=np.float32),
                                     shape=(self.lenObs,))
        self._device = device
        self._vec = None

    def dataToState(self, systemState):
        """dataToState (6DoF.py:467-483 / 3DoF.py:397-409) evaluated for an arbitrary system state."""
        v = self._vec
        saved = v._state[:, 0].clone()
        v._state[:, 0] = torch.as_tensor(np.asarray(systemState, dtype=np.float64), device=v.device)
        obs = v.observe()[0].cpu().numpy()
        v._state[:, 0] = saved
        return obs

    def _sync_and_log(self):
        sp = self._sync_from_device()
        veh = self.vehicle
        self.timeHistory.append(np.concatenate([[self.time], self.systemState, veh.generalisedControlForces, veh.controlVector, sp]))

    def reset(self, initialSetpoint=None):
        if self._vec is None:
            self._vec = self._VEC(1, seed=0 if self.seed is None else int(self.seed), dt=self.dt, maxSteps=self._max_episode_steps,
                                  n_sub=self.nSub, action_mode="setpoint", dtype=torch.float64, device=self._device,
                                  auto_reset=False, record_aux=True)
        self.iStep = 0
        self.time = 0.
        self.iWp = 0
        self._vec.reset(initialSetpoint=initialSetpoint)
        self.fixedSp = self._vec.fixedSp
        self._new_vehicle(self._vec.setPoint[0].cpu().numpy())
        self.timeHistory = []
        self._sync_and_log()
        self.steps_beyond_done = 0
        return self.state

    def step(self, action):
        self.iStep += 1
        self.time += self.dt
        a = torch.as_tensor(np.asarray(action, dtype=np.float64).reshape(1, self.lenAction), device=self._vec.device)
        _, _, done, _ = self._vec.step(a)
        done = bool(done[0])
        self._sync_and_log()
        reward = 0.
        if done:
            import pandas
            self.timeHistory = pandas.DataFrame(data=np.array(self.timeHistory), columns=self._VEC.HISTORY_COLUMNS)
            self.steps_beyond_done += 1
        else:
            self.steps_beyond_done = 0
        return self.state, reward, done, {}
