"""The callers and data formats either side of the env-step path (SURVEY.md 8(f), rows N1 / N2):

* ``TrajectoryRecorder`` - per-step ``timeHistory`` rows of the first k environments kept on the device and
  exported with the reference's column names (6DoF.py:578-587, 3DoF.py:498-508,
  tag_00.../verySimpleAuv.py:389-401) / as the ``ep_<i>.csv`` files ``evaluate_agent`` writes
  (resources.py:175-178);
* ``evaluate_agent`` - the reference's evaluation loop (resources.py:145-198) for single and batched envs;
* ``Sb3VecEnv`` - numpy-facing adapter with the Stable-Baselines3 ``VecEnv`` protocol the legacy training
  scripts drive (tag_00.../main_00_sbl.py:145-146), including ``VecMonitor``'s ``r,l,t`` CSV;
* ``SymmetryReplayBuffer`` - the mirror-image augmenting replay buffer of
  tag_00.../main_02_sbl_contrib_customBuffer.py:57-160, filled on the device by ``mvrl_replay_add_symmetric``;
* ``ReplayBuffer`` - SB3 2.x's plain ``ReplayBuffer`` (the buffer of SAC / TQC, legacy/main_00_sbl.py) filled from and sampled
  on the device, one kernel per ``add`` (``mvrl_replay_add``) and per ``sample`` (``mvrl_replay_sample``);
* ``EnvBlocks`` - a batched env stepped as independent blocks of environments, each block a chain of launches on its own
  stream: what the ``SubprocVecEnv`` workers of the legacy scripts are to each other (tag_00.../main_00_sbl.py:145-146,
  script_0_checkScaling.py:23-40); ``EnvShards`` - the same for separate env objects of any kind.
"""
import collections
import csv
import ctypes as C
import json
import os
import time

import numpy as np
import torch

from . import _lib
from ._gymshim import Box
from .rov6 import _RovVecEnv


class EnvBlocks:
    """Step a batched 6DoF env as ``groups`` independent blocks of environments, block ``g`` on its own CUDA stream.

    The reference scales by running ``nProc`` workers that step their environments without waiting for each other
    (``SubprocVecEnv([make_env(i) for i in range(nProc)])``, tag_00.../main_00_sbl.py:145-146; its scaling check,
    script_0_checkScaling.py:23-40, times exactly that).  On the GPU the same independence pays differently: one launch
    per step leaves the SMs under-used while its first CTAs load and its last ones store (a 131 072-environment step is
    1.15 waves of CTAs: 30.2 us), whereas chains of smaller launches on separate streams drift out of phase, so one
    block's prologue / epilogue runs under the other blocks' RK4 loops (four blocks: 22.8 us, the rate of a 1 Mi-env
    launch; profiles/r2_zz_stream_groups.jsonl).  Results do not depend on the blocking: every block runs the same kernel on
    its own environments (``mvrl_rov6_step_range``), random draws are keyed on the global environment id.

        blocks = EnvBlocks(env, 4)
        with blocks:                       # fork: the block streams wait for the caller's stream
            for k in range(K):
                blocks.step_async()        # block g's k-th step queues behind its own (k-1)-th only
        # join: the caller's stream waits for every block - env.obs / env.systemState are complete from here on

    ``for lo, cnt, stream in blocks:`` gives the caller the blocks to queue its own per-block work (a policy) on.
    Works eagerly and inside CUDA-graph capture (the block streams fork from and re-join the capturing stream).
    ``align``: block starts are multiples of it (2 keeps the two-environments-per-thread kernel's 8-byte row alignment;
    128 = the rollout actor's tile)."""

    def __init__(self, env, groups, align=2):
        if not hasattr(env, "step_range_async"):
            raise TypeError("EnvBlocks needs a batched env with step_range_async (the 6DoF VecEnv); use EnvShards for separate env objects")
        groups, align = int(groups), int(align)
        if groups < 1 or align < 1:
            raise ValueError("groups and align must be positive")
        self.env = env
        n = env.num_envs
        per = -(-n // groups)
        per += (-per) % align
        self.blocks = [(lo, min(per, n - lo)) for lo in range(0, n, per)]
        self._init_streams(env.device, len(self.blocks))

    def _init_streams(self, device, count):
        self.device = device
        self.streams = [torch.cuda.Stream(device=device) for _ in range(count)]
        self._forked = False

    def __len__(self):
        return len(self.streams)

    def __iter__(self):
        return iter([(lo, cnt, s) for (lo, cnt), s in zip(self.blocks, self.streams)])

    def fork(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            s.wait_stream(cur)
        self._forked = True

    def join(self):
        cur = torch.cuda.current_stream(self.device)
        for s in self.streams:
            cur.wait_stream(s)
        self._forked = False

    def __enter__(self):
        self.fork()
        return self

    def __exit__(self, *exc):
        self.join()
        return False

    def _require_fork(self):
        if not self._forked:
            raise RuntimeError("%s.step_async outside fork() / join() (use `with blocks:`)" % type(self).__name__)

    def step_async(self):
        """Queue one env step of every block on its stream (actions are read from the env's action buffer)."""
        self._require_fork()
        for (lo, cnt), s in zip(self.blocks, self.streams):
            with torch.cuda.stream(s):
                self.env.step_range_async(lo, cnt)


class EnvShards(EnvBlocks):
    """The same for SEPARATE env objects of any kind (6DoF, 3DoF, legacy) - literally the reference's list of workers, each
    with its own buffers: ``EnvShards([AuvVecEnv(n // 4, flow, env_id0=i * (n // 4), ...) for i in range(4)])``.  Shards
    created with consecutive ``env_id0`` draw the same random numbers as one env over all of them (tested bitwise), and
    each steps as a chain on its own stream.  ``for env, stream in shards:`` to queue per-shard work."""

    def __init__(self, envs):
        self.envs = list(envs)
        if not self.envs:
            raise ValueError("EnvShards needs at least one env")
        self._init_streams(self.envs[0].device, len(self.envs))

    def __iter__(self):
        return iter(list(zip(self.envs, self.streams)))

    def step_async(self):
        """Queue one env step of every shard on its stream (each reads its own action buffer)."""
        self._require_fork()
        for e, s in zip(self.envs, self.streams):
            with torch.cuda.stream(s):
                e.step_async()


class TrajectoryRecorder:
    """Keeps the reference's per-step log rows of environments ``0 .. num_record-1`` in a device buffer
    ``[capacity, columns, num_record]`` (written by device-to-device copies of the SoA buffers, no host
    round trip per step) and turns them into pandas DataFrames / CSV files on demand.  The env must have been
    built with ``record_aux=True`` (controller forces, rpm / force terms live in ``aux``).

    Rows belong to the episode in progress: ``on_reset`` starts a new one, ``on_step`` appends one row per
    environment.  With auto-reset envs, per-environment row counts restart when that environment terminates."""

    def __init__(self, env, num_record=1, capacity=None):
        if getattr(env, "HISTORY_COLUMNS", None) is None:
            raise TypeError("unsupported env type %s: a batched env with HISTORY_COLUMNS expected" % type(env).__name__)
        self.env, self._rov = env, isinstance(env, _RovVecEnv)
        if env._aux is None:
            raise ValueError("build the env with record_aux=True to record trajectories")
        self.k = min(int(num_record), env.num_envs)
        self.columns = env.HISTORY_COLUMNS
        self.capacity = int(capacity if capacity is not None else env._max_episode_steps + 1)
        self.buf = torch.zeros((self.capacity, len(self.columns), self.k), dtype=env.dtype, device=env.device)
        self.count = torch.zeros(self.k, dtype=torch.long, device=env.device)
        self._rows = torch.arange(self.k, device=env.device)
        self._last_actions = None

    def _row(self):
        e, k = self.env, self.k
        t = (e._istep[:k].to(e.dtype) * e.dt).unsqueeze(0)
        if self._rov:
            return torch.cat([t, e._state[:, :k], e._aux[:, :k], e._setpoint[:, :k]])
        s, aux = e._state[:, :k], e._aux[:, :k]
        zeros = e.positionTarget[:k].T if hasattr(e, "positionTarget") else torch.zeros((2, k), dtype=e.dtype, device=e.device)
        act = self._last_actions if self._last_actions is not None else torch.zeros((3, k), dtype=e.dtype, device=e.device)
        return torch.cat([e._istep[:k].to(e.dtype).unsqueeze(0), t, e._reward[:k].unsqueeze(0), s[0:3], zeros, e._target[0:1, :k],
                          aux[0:6], s[3:6], aux[6:9], aux[9:14], act, e._obs[:, :k]])

    def on_reset(self):
        """Call after ``env.reset()``: the 3DoF / 6DoF logs start with the initial row (6DoF.py:522-524)."""
        self.count.zero_()
        if self._rov:
            self._append(self._row(), torch.ones(self.k, dtype=torch.bool, device=self.env.device))

    def _append(self, row, mask):
        idx = self.count.clamp(max=self.capacity - 1)
        cur = self.buf[idx, :, self._rows]                      # [k, C]
        self.buf[idx, :, self._rows] = torch.where(mask.unsqueeze(1), row.T, cur)
        self.count += mask.long()

    def on_step(self, actions=None):
        """Call after ``env.step``.  For auto-reset envs the row of a terminating environment is the reset
        state (the terminal state itself is not kept by the env); its counter restarts."""
        e, k = self.env, self.k
        if actions is not None:   # [N, A] (or feature-major [A, N])
            a = actions.T if tuple(actions.shape) == (e.num_envs, e.lenAction) else actions
            self._last_actions = a[:, :k].to(device=e.device, dtype=e.dtype)
        done = e._done[:k].bool()
        fresh = done & bool(e.auto_reset)
        self.count = torch.where(fresh, torch.zeros_like(self.count), self.count)
        self._append(self._row(), torch.ones(k, dtype=torch.bool, device=e.device))

    def dataframe(self, i=0):
        import pandas
        n = int(self.count[i])
        return pandas.DataFrame(self.buf[:n, :, i].cpu().numpy().astype(float), columns=self.columns)

    def to_csv(self, save_dir, prefix="ep"):
        """One ``<prefix>_<i>.csv`` per recorded environment, like ``evaluate_agent(saveDir=...)`` (resources.py:175-178)."""
        os.makedirs(save_dir, exist_ok=True)
        paths = []
        for i in range(self.k):
            p = os.path.join(save_dir, "%s_%d.csv" % (prefix, i))
            self.dataframe(i).to_csv(p, index=False)
            paths.append(p)
        return paths


def evaluate_agent(agent, env, num_episodes=1, num_steps=None, deterministic=True, num_last_for_reward=None,
                   render=False, init=None, saveDir=None):
    """resources.py:145-198 / tag_00.../resources.py:49-101.  ``agent`` is anything with the SB3-like
    ``predict(obs, deterministic) -> (action, state)``.

    * single-vehicle envs (the reference-shaped ``AuvEnv`` / ``BlueROV2Heavy*Env``): same loop and return value
      as the reference - (mean, median, list of episode rewards); ``saveDir`` gets ``ep_<i>.csv``.
    * batched ``*VecEnv``: every environment runs ``num_episodes`` episodes at once (auto-reset must be off or
      ``num_episodes == 1``); episode rewards are per environment."""
    if saveDir is not None:
        os.makedirs(saveDir, exist_ok=True)
    batched = hasattr(env, "num_envs")
    all_rewards = []
    if num_steps is None:
        num_steps = 1000000
    for i_ep in range(num_episodes):
        if batched:
            obs = env.reset()
            total = torch.zeros(env.num_envs, dtype=torch.float64, device=env.device)
            alive = torch.ones(env.num_envs, dtype=torch.bool, device=env.device)
            for _ in range(min(num_steps, env._max_episode_steps)):
                action, _ = agent.predict(obs, deterministic=deterministic)
                obs, reward, done, _ = env.step(action)
                total += torch.where(alive, reward.to(torch.float64), torch.zeros_like(total))
                alive &= ~done
                if not bool(alive.any()):
                    break
            all_rewards.extend(total.cpu().tolist())
            continue
        try:
            obs = env.reset(fixedInitialValues=init, keepTimeHistory=saveDir is not None)
        except TypeError:   # the 3DoF / 6DoF envs take reset(initialSetpoint=None)
            obs = env.reset(init) if init is not None else env.reset()
        rewards = []
        for _ in range(num_steps):
            action, _ = agent.predict(obs, deterministic=deterministic)
            obs, reward, done, _ = env.step(action)
            rewards.append(reward)
            if done:
                if saveDir is not None:
                    env.timeHistory.to_csv(os.path.join(saveDir, "ep_{:d}.csv".format(i_ep)), index=False)
                break
        all_rewards.append(sum(rewards) if num_last_for_reward is None else float(np.mean(rewards[-num_last_for_reward:])))
    mean, median = float(np.mean(all_rewards)), float(np.median(all_rewards))
    print("  Mean reward:  ", mean)
    print("  Median reward:", median)
    print("  Num episodes: ", num_episodes)
    return mean, median, all_rewards


class Sb3VecEnv:
    """Stable-Baselines3 ``VecEnv`` protocol over a batched device env: numpy float32 observations / rewards /
    dones, a list of per-env info dicts with ``terminal_observation`` and (``VecMonitor`` behaviour)
    ``episode = {"r", "l", "t"}`` for the environments that finished, optional ``<filename>.monitor.csv``.
    What ``SubprocVecEnv([make_env(i) ...]) + VecMonitor`` provides in tag_00.../main_00_sbl.py:145-146 - one
    process, one kernel launch per step instead of nProc worker processes and pipes."""

    def __init__(self, env, monitor_file=None, flag_time_limit=False):
        """``flag_time_limit``: add ``TimeLimit.truncated`` to the info of an episode that ended by reaching ``maxSteps``
        while inside the bounds.  Off by default: the reference envs set ``done`` themselves (no ``TimeLimit`` wrapper), so
        upstream the key never exists and SB3's off-policy learners do not bootstrap through max-step terminations."""
        self.env = env
        self.flag_time_limit = bool(flag_time_limit)
        self.num_envs = env.num_envs
        self.observation_space = Box(-1.0, 1.0, shape=(env.lenObs,), dtype=np.float32)
        self.action_space = Box(-1.0, 1.0, shape=(env.lenAction,), dtype=np.float32)
        self._actions = None
        self._ret = np.zeros(self.num_envs, dtype=np.float64)
        self._len = np.zeros(self.num_envs, dtype=np.int64)
        self._t0 = time.time()
        self._csv = None
        if monitor_file is not None:
            path = monitor_file if monitor_file.endswith("monitor.csv") else monitor_file + ".monitor.csv"
            os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
            self._fh = open(path, "w", newline="")
            self._fh.write("#%s\n" % json.dumps({"t_start": self._t0, "env_id": type(env).__name__}))
            self._csv = csv.DictWriter(self._fh, fieldnames=("r", "l", "t"))
            self._csv.writeheader()

    def reset(self):
        self._ret[:] = 0
        self._len[:] = 0
        return self.env.reset().to(torch.float32).cpu().numpy()

    def step_async(self, actions):
        self._actions = torch.as_tensor(np.asarray(actions), dtype=self.env.dtype, device=self.env.device)

    def step_wait(self):
        obs, rew, done, info = self.env.step(self._actions)
        obs_np = obs.to(torch.float32).cpu().numpy()
        rew_np = rew.to(torch.float32).cpu().numpy()
        done_np = done.cpu().numpy()
        self._ret += rew_np
        self._len += 1
        infos = [{} for _ in range(self.num_envs)]
        idx = np.nonzero(done_np)[0]
        if idx.size:
            term = info.get("terminal_observation")
            term_np = term[torch.as_tensor(idx, device=term.device)].to(torch.float32).cpu().numpy() if term is not None else None
            now = round(time.time() - self._t0, 6)
            for j, i in enumerate(idx):
                ep = {"r": round(float(self._ret[i]), 6), "l": int(self._len[i]), "t": now}
                infos[i]["episode"] = ep
                if self.flag_time_limit and self._len[i] >= self.env._max_episode_steps and not self._ended_by_bounds(i, done_np):
                    infos[i]["TimeLimit.truncated"] = True
                if term_np is not None:
                    infos[i]["terminal_observation"] = term_np[j]
                if self._csv is not None:
                    self._csv.writerow(ep)
            if self._csv is not None:
                self._fh.flush()
            self._ret[idx] = 0
            self._len[idx] = 0
        return obs_np, rew_np, done_np, infos

    def _ended_by_bounds(self, i, done_np):
        """True when environment ``i`` terminated by leaving the domain (legacy envs: verySimpleAuv.py:332-345) rather
        than by the step limit; the rov envs have no bounds termination."""
        oob = getattr(self.env, "out_of_bounds", None)
        return bool(oob[i]) if oob is not None else False

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        if self._csv is not None:
            self._fh.close()
            self._csv = None

    def seed(self, seed=None):
        return [None] * self.num_envs

    def get_attr(self, attr_name, indices=None):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        return [getattr(self.env, attr_name)] * n

    def set_attr(self, attr_name, value, indices=None):
        setattr(self.env, attr_name, value)

    def env_method(self, method_name, *args, indices=None, **kwargs):
        return [getattr(self.env, method_name)(*args, **kwargs)]

    def env_is_wrapped(self, wrapper_class, indices=None):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        return [False] * n

    def render(self, mode="human"):
        return None


class SymmetryReplayBuffer:
    """``CustomReplayBuffer`` of tag_00.../main_02_sbl_contrib_customBuffer.py:57-160 on the device: every
    ``add`` stores the batch of transitions of the legacy env plus its four mirror images in consecutive
    slots, until the buffer has rolled over more than twice; then only the real transitions.  ``add`` takes
    the env's feature-major buffers directly (no transposes, no host copy).

    ``buffer_size`` counts TRANSITIONS like upstream: SB3's ``ReplayBuffer.__init__`` (the base class the reference
    subclasses) keeps ``max(buffer_size // n_envs, 1)`` slots of ``n_envs`` transitions each, and so does this class
    (attribute ``buffer_size`` = slots afterwards, as in SB3).  ``timeouts`` holds the ``TimeLimit.truncated`` flags
    (``handle_timeout_termination=True`` is hard-wired upstream, :72-73)."""
    N_TRANSFORMS = 5

    def __init__(self, buffer_size, n_envs, dtype=torch.float32, device="cuda", ld=None):
        self.n_envs = int(n_envs)
        self.buffer_size = max(int(buffer_size) // self.n_envs, 1)
        if self.buffer_size < self.N_TRANSFORMS:
            # upstream would overwrite the same slot several times within one add(); the five images of an add are written
            # by one launch here, so they need five distinct slots
            raise ValueError("buffer_size // n_envs = %d slots: need at least %d (one per mirror image)" % (self.buffer_size, self.N_TRANSFORMS))
        self.dtype, self.device = dtype, torch.device(device)
        self.ld = int(ld) if ld is not None else self.n_envs
        z = lambda *shape, dt=dtype: torch.zeros(shape, dtype=dt, device=self.device)
        self.observations, self.next_observations = z(self.buffer_size, self.n_envs, 11), z(self.buffer_size, self.n_envs, 11)
        self.actions, self.rewards = z(self.buffer_size, self.n_envs, 3), z(self.buffer_size, self.n_envs)
        self.dones = z(self.buffer_size, self.n_envs, dt=torch.uint8)
        self.timeouts = z(self.buffer_size, self.n_envs, dt=torch.uint8)
        self.pos, self.full, self.nRollovers = 0, False, 0

    def add(self, obs_fm, next_obs_fm, action_fm, reward, done, timeouts=None):
        """obs_fm / next_obs_fm ``[11, ld]``, action_fm ``[3, ld]``, reward ``[>= n]``, done uint8 ``[>= n]``;
        ``timeouts`` (optional, uint8 / bool ``[>= n]``, or the list of ``infos`` dicts of a ``VecEnv.step``): the
        ``TimeLimit.truncated`` flags, all false when omitted."""
        lib = _lib.load()
        # position bookkeeping exactly as upstream (:139-160): the roll-over test sits inside the loop over the
        # transformations, so the mirror images stop in the middle of an add() when the third roll-over happens
        pos0, nt = self.pos, 0
        for i in range(self.N_TRANSFORMS):
            if self.nRollovers > 2 and i != 0:
                continue
            nt += 1
            self.pos += 1
            if self.pos == self.buffer_size:
                self.full, self.pos = True, 0
                self.nRollovers += 1
        done = done if done.dtype == torch.uint8 else done.to(torch.uint8)
        if timeouts is not None:
            if isinstance(timeouts, (list, tuple)):   # infos, as upstream's add() receives them (:150-151)
                timeouts = np.array([bool(i.get("TimeLimit.truncated", False)) for i in timeouts], dtype=np.uint8)
            timeouts = torch.as_tensor(timeouts, device=self.device)
            timeouts = timeouts if timeouts.dtype == torch.uint8 else timeouts.to(torch.uint8)
        _lib.check(lib.mvrl_replay_add_symmetric(
            _lib.torch_dtype_code(self.dtype), self.n_envs, obs_fm.stride(0), _lib.ptr(obs_fm), _lib.ptr(next_obs_fm), _lib.ptr(action_fm),
            _lib.ptr(reward), _lib.ptr(done), _lib.ptr(timeouts), _lib.ptr(self.observations), _lib.ptr(self.next_observations),
            _lib.ptr(self.actions), _lib.ptr(self.rewards), _lib.ptr(self.dones), _lib.ptr(self.timeouts), self.buffer_size, pos0, nt,
            _lib.current_stream(self.device)))

    def size(self):
        return self.buffer_size if self.full else self.pos

    def sample(self, batch_size, generator=None):
        """Uniform sample of stored (slot, env) pairs -> dict of ``[batch, k]`` tensors."""
        slot = torch.randint(0, self.size(), (batch_size,), device=self.device, generator=generator)
        env = torch.randint(0, self.n_envs, (batch_size,), device=self.device, generator=generator)
        return {"observations": self.observations[slot, env], "next_observations": self.next_observations[slot, env],
                "actions": self.actions[slot, env], "rewards": self.rewards[slot, env], "dones": self.dones[slot, env],
                "timeouts": self.timeouts[slot, env]}


ReplayBufferSamples = collections.namedtuple("ReplayBufferSamples", ["observations", "actions", "next_observations", "dones", "rewards"])
ReplayBufferSamples.__doc__ = "SB3's ``ReplayBufferSamples`` fields as device tensors in the env's dtype; ``dones`` = done * (1 - timeout)."


def _timeout_mask(timeouts, n, device):
    """``None``, a bool / uint8 tensor ``[n]`` or the list of info dicts of a ``VecEnv.step`` -> uint8 ``[n]`` on ``device``
    (or None): the ``TimeLimit.truncated`` flags SB3's ``ReplayBuffer.add`` reads from the infos."""
    if timeouts is None:
        return None
    if isinstance(timeouts, (list, tuple)):
        if len(timeouts) != n:
            raise ValueError("timeouts: %d info dicts for %d environments" % (len(timeouts), n))
        timeouts = np.array([bool(i.get("TimeLimit.truncated", False)) for i in timeouts], dtype=np.uint8)
    t = torch.as_tensor(timeouts, device=device)
    if t.dtype not in (torch.bool, torch.uint8) or t.dim() != 1 or t.shape[0] != n:
        raise ValueError("timeouts must be a bool / uint8 tensor [%d] or a list of info dicts, got %s %s" % (n, t.dtype, tuple(t.shape)))
    return t.to(torch.uint8).contiguous()


class ReplayBuffer:
    """Stable-Baselines3 2.x ``ReplayBuffer`` (``optimize_memory_usage=False``, ``handle_timeout_termination=True``) on the
    device, filled straight from a batched env's feature-major buffers - what SAC / TQC's ``OffPolicyAlgorithm.
    _store_transition`` followed by ``ReplayBuffer.add`` stores, and ``ReplayBuffer.sample`` draws from:

        buf = ReplayBuffer(buffer_size, env, seed=0)
        env.reset(); buf.on_reset(env)            # SB3: self._last_obs = env.reset()
        for t in range(T):                        # eagerly, or captured as one CUDA graph and replayed
            pol.act(env); env.step_async(); buf.add(env)
        batch = buf.sample(256)                   # ReplayBufferSamples of device tensors

    ``buffer_size`` counts transitions: ``max(buffer_size // n_envs, 1)`` slots of ``n_envs`` transitions.  ``observations``
    / ``next_observations`` ``[slots, n_envs, obs_dim]``, ``actions [slots, n_envs, act_dim]``, ``rewards [slots, n_envs]``
    in the env's dtype (bit copies of what the env produced); ``dones`` / ``timeouts [slots, n_envs]`` uint8.

    ``add`` stores the observation the actor saw (kept in the staging row ``last_obs [obs_dim, ld]``, SB3's ``_last_obs``,
    because the step overwrites the env's obs), the env's action buffer, reward and done, and as ``next_obs`` the terminal
    observation where an environment was auto-reset, else the post-step obs; then the staging row takes the post-step obs.
    After an explicit ``env.reset()`` (masked or not) call ``on_reset(env)``.

    Slot position, number of adds and number of ``sample`` calls live in the int64 device tensor ``cursor``; the kernels read
    and advance it, so T adds and samples captured in a CUDA graph and replayed R times behave like T * R eager calls, and
    every ``sample`` (eager call or replay) draws new indices: Philox4x32-10 stream 9 keyed on (``seed``, sample index, call
    number).  ``size()``, ``pos`` and ``full`` read the cursor (they synchronise).  One buffer per env; with ``EnvShards``,
    one per shard.

    ``cursor`` = [pos, adds, sample calls, pos << 32, 0] between launches: the add kernel takes pos and its block ticket from
    the packed word ``cursor[3]`` in one atomic (``include/mvrl.h``), ``cursor[0]`` is the copy the sampler and the host read,
    and pos = adds mod slots.  ``load_state_dict`` refuses a cursor that breaks any of this."""

    def __init__(self, buffer_size, env, seed=0):
        self.n_envs, self.obs_dim, self.act_dim = int(env.num_envs), int(env.lenObs), int(env.lenAction)
        if int(buffer_size) < 1:
            raise ValueError("buffer_size must be >= 1 (a buffer needs at least one slot)")
        if self.n_envs < 1:
            raise ValueError("the env has no environments")
        if not (1 <= self.obs_dim <= _lib.REPLAY_MAX_DIM and 1 <= self.act_dim <= _lib.REPLAY_MAX_DIM):
            raise ValueError("obs_dim %d / act_dim %d: the replay kernels take 1 .. %d" % (self.obs_dim, self.act_dim, _lib.REPLAY_MAX_DIM))
        self.dtype_code = _lib.torch_dtype_code(env.dtype)
        _lib.require_cuda()
        self.buffer_size = max(int(buffer_size) // self.n_envs, 1)
        self.dtype, self.device, self.ld, self.seed = env.dtype, env.device, int(env.ld), int(seed)
        z = lambda *shape, dt=self.dtype: torch.zeros(shape, dtype=dt, device=self.device)
        s, n = self.buffer_size, self.n_envs
        self.observations, self.next_observations = z(s, n, self.obs_dim), z(s, n, self.obs_dim)
        self.actions, self.rewards = z(s, n, self.act_dim), z(s, n)
        self.dones, self.timeouts = z(s, n, dt=torch.uint8), z(s, n, dt=torch.uint8)
        self.last_obs = z(self.obs_dim, self.ld)
        self.cursor = z(5, dt=torch.int64)     # pos, adds, sample calls, pos << 32 | add blocks, sample blocks (mvrl.h)
        self._adds = 0                         # host count: only to refuse sampling an empty buffer
        self._storage = _lib.MvrlReplayStorage(*[t.data_ptr() for t in (
            self.observations, self.next_observations, self.actions, self.rewards, self.dones, self.timeouts, self.last_obs, self.cursor)])

    def _check_env(self, env):
        if (int(env.num_envs), int(env.lenObs), int(env.lenAction), env.dtype, env.device, int(env.ld)) != \
                (self.n_envs, self.obs_dim, self.act_dim, self.dtype, self.device, self.ld):
            raise ValueError("env (n %d, obs %d, act %d, %s, %s, ld %d) does not match the buffer (n %d, obs %d, act %d, %s, %s, ld %d)"
                             % (env.num_envs, env.lenObs, env.lenAction, env.dtype, env.device, env.ld,
                                self.n_envs, self.obs_dim, self.act_dim, self.dtype, self.device, self.ld))
        if env.auto_reset and env._terminal_obs is None:
            raise ValueError("the env auto-resets but keeps no terminal observation (record_terminal_obs=False): next_obs of a "
                             "finished episode would be the reset observation")

    def on_reset(self, env):
        """SB3's ``self._last_obs = env.reset()``: copy the env's obs into the staging row (after any ``env.reset()``)."""
        self._check_env(env)
        self.last_obs.copy_(env._obs)

    def add(self, env, timeouts=None):
        """Store the transition of the env step just queued (one launch on the current stream, no synchronisation).
        ``timeouts``: ``TimeLimit.truncated`` flags as a bool / uint8 tensor ``[n_envs]`` or the list of info dicts; all
        false when omitted (the reference envs have no ``TimeLimit`` wrapper)."""
        self._check_env(env)
        t = _timeout_mask(timeouts, self.n_envs, self.device)
        _lib.check(_lib.load().mvrl_replay_add(
            self.dtype_code, self.n_envs, self.ld, self.obs_dim, self.act_dim, self.buffer_size, C.byref(self._storage),
            _lib.ptr(env._obs), _lib.ptr(env._terminal_obs), _lib.ptr(env._action), _lib.ptr(env._reward), _lib.ptr(env._done),
            _lib.ptr(t), _lib.current_stream(self.device)))
        self._adds += 1

    def sample(self, batch_size):
        """``ReplayBuffer.sample(batch_size)``: slot uniform in ``[0, size())``, environment uniform in ``[0, n_envs)``.
        Returns ``ReplayBufferSamples`` of new device tensors ``[B, obs_dim]``, ``[B, act_dim]``, ``[B, obs_dim]``,
        ``[B, 1]``, ``[B, 1]`` (one launch, no synchronisation)."""
        b = int(batch_size)
        if b < 1 or b >= 2 ** 31:
            raise ValueError("batch_size must be in [1, 2^31), got %d" % b)
        if self._adds == 0:
            raise ValueError("sample() on an empty replay buffer")
        e = lambda *shape: torch.empty(shape, dtype=self.dtype, device=self.device)
        out = ReplayBufferSamples(e(b, self.obs_dim), e(b, self.act_dim), e(b, self.obs_dim), e(b, 1), e(b, 1))
        _lib.check(_lib.load().mvrl_replay_sample(
            self.dtype_code, self.n_envs, self.obs_dim, self.act_dim, self.buffer_size, C.byref(self._storage), b,
            self.seed & (2 ** 64 - 1), _lib.ptr(out.observations), _lib.ptr(out.actions), _lib.ptr(out.next_observations),
            _lib.ptr(out.dones), _lib.ptr(out.rewards), _lib.current_stream(self.device)))
        return out

    @property
    def pos(self):
        return int(self.cursor[0])

    @property
    def full(self):
        return int(self.cursor[1]) >= self.buffer_size

    def size(self):
        """Number of filled slots (SB3: ``buffer_size if full else pos``); reads the device cursor."""
        c = self.cursor[:2].tolist()
        return self.buffer_size if c[1] >= self.buffer_size else c[0]

    _STATE = ("observations", "next_observations", "actions", "rewards", "dones", "timeouts", "last_obs", "cursor")

    def state_dict(self):
        """Storage, staging row and cursor (copies) - what ``save_replay_buffer`` keeps."""
        d = {k: getattr(self, k).clone() for k in self._STATE}
        d["seed"] = self.seed
        return d

    def load_state_dict(self, d):
        """Copy a ``state_dict`` into this buffer's tensors in place (a captured graph keeps working on them)."""
        pos, adds, calls, word, sticket = [int(v) for v in torch.as_tensor(d["cursor"]).reshape(-1)[:5].tolist()]
        if not (adds >= 0 and calls >= 0 and pos == adds % self.buffer_size and word == pos << 32 and sticket == 0):
            raise ValueError("cursor %s is not [pos, adds, calls, pos << 32, 0] with pos = adds mod %d"
                             % ([pos, adds, calls, word, sticket], self.buffer_size))
        for k in self._STATE:
            src = torch.as_tensor(d[k])
            dst = getattr(self, k)
            if tuple(src.shape) != tuple(dst.shape) or src.dtype != dst.dtype:
                raise ValueError("%s: %s %s does not match the buffer's %s %s" % (k, src.dtype, tuple(src.shape), dst.dtype, tuple(dst.shape)))
            dst.copy_(src)
        self.seed = int(d["seed"])
        self._adds = int(self.cursor[1])
