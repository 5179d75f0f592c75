"""GPU: vec_tools.ReplayBuffer (kernels replay_add_kernel / replay_sample_kernel) against a NumPy restatement of
Stable-Baselines3 2.x's ReplayBuffer fed by OffPolicyAlgorithm._store_transition, bit for bit, on every batched env; the
sampler against the NumPy Philox restatement; uniformity; CUDA-graph replay against an eager twin; state_dict; the size the
benchmark times; and the argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch

from conftest import load_golden
from test_replay_cpu import replay_sample_indices

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import (AuvCylVecEnv, AuvVecEnv, BlueROV2Heavy3DoFVecEnv, BlueROV2Heavy6DoFVecEnv,
                                                         ReplayBuffer, SquashedGaussianPolicy, _lib)
    from marinevehiclereinforcementlearning_b200.tag_00_Dec2023_simpleControlTurbulence import flowGenerator

DEV = "cuda"


# ---- SB3 2.x, restated (stable_baselines3/common/buffers.py, common/off_policy_algorithm.py) ---------------------------
class Sb3ReplayBuffer:
    """``ReplayBuffer`` with ``optimize_memory_usage=False``, ``handle_timeout_termination=True``: ``__init__`` and ``add``.
    Storage dtypes are the device buffer's (SB3 keeps rewards / dones / timeouts as float32; the values stored here are the
    env's rewards and 0 / 1 flags, copied bit for bit)."""

    def __init__(self, buffer_size, obs_dim, act_dim, n_envs, dtype):
        self.buffer_size = max(buffer_size // n_envs, 1)
        self.n_envs, self.pos, self.full = n_envs, 0, False
        self.observations = np.zeros((self.buffer_size, n_envs, obs_dim), dtype=dtype)
        self.next_observations = np.zeros((self.buffer_size, n_envs, obs_dim), dtype=dtype)
        self.actions = np.zeros((self.buffer_size, n_envs, act_dim), dtype=dtype)
        self.rewards = np.zeros((self.buffer_size, n_envs), dtype=dtype)
        self.dones = np.zeros((self.buffer_size, n_envs), dtype=np.uint8)
        self.timeouts = np.zeros((self.buffer_size, n_envs), dtype=np.uint8)

    def add(self, obs, next_obs, action, reward, done, infos):
        self.observations[self.pos] = np.array(obs)
        self.next_observations[self.pos] = np.array(next_obs)
        self.actions[self.pos] = np.array(action)
        self.rewards[self.pos] = np.array(reward)
        self.dones[self.pos] = np.array(done)
        self.timeouts[self.pos] = np.array([info.get("TimeLimit.truncated", False) for info in infos])
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True
            self.pos = 0

    def size(self):
        return self.buffer_size if self.full else self.pos


def store_transition(buf, last_obs, new_obs, buffer_action, reward, dones, infos):
    """``OffPolicyAlgorithm._store_transition``: next_obs = new_obs with ``terminal_observation`` where done; returns the
    new ``_last_obs``."""
    next_obs = new_obs.copy()
    for i, done in enumerate(dones):
        if done and infos[i].get("terminal_observation") is not None:
            next_obs[i] = infos[i]["terminal_observation"]
    buf.add(last_obs, next_obs, buffer_action, reward, dones, infos)
    return new_obs


# ---- envs ---------------------------------------------------------------------------------------------------------
def make_flow(dtype):
    g = load_golden("legacy")
    base = g["ltm"][None] + 0.05 * np.random.default_rng(7).standard_normal((int(g["nt"]),) + g["ltm"].shape)
    return flowGenerator.ReconstructedFlow.from_base_field(base, float(g["base_dx"]), float(g["base_dy"]), float(g["base_dt"]),
                                                           dtype=dtype, device=DEV)


ENVS = {   # name -> (constructor(n), action scale)
    "rov6_setpoint_f32": (lambda n: BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, maxSteps=4, seed=3), 1.0),
    "rov6_rpm_f64": (lambda n: BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", dtype=torch.float64, device=DEV, maxSteps=3, seed=4), 3500.0),
    "rov6_force_f32": (lambda n: BlueROV2Heavy6DoFVecEnv(n, action_mode="force", dtype=torch.float32, device=DEV, maxSteps=5, seed=5), 20.0),
    "rov6_force_f32_no_auto_reset": (lambda n: BlueROV2Heavy6DoFVecEnv(n, action_mode="force", dtype=torch.float32, device=DEV,
                                                                       maxSteps=4, seed=5, auto_reset=False), 20.0),
    "rov3": (lambda n: BlueROV2Heavy3DoFVecEnv(n, dtype=torch.float32, device=DEV, maxSteps=4, seed=6), 1.0),
    "auv_noise": (lambda n: AuvVecEnv(n, make_flow(torch.float64), dtype=torch.float64, maxSteps=5, seed=7,
                                      noiseMagCoeffs=0.1, noiseMagActuation=0.1), 1.0),
    "auv_cyl": (lambda n: AuvCylVecEnv(n, make_flow(torch.float32), dtype=torch.float32, maxSteps=3, seed=8), 1.0),
}


def host_fm(t, n):
    return t[:, :n].T.cpu().numpy()


def same_bits(t, a):
    """torch tensor == numpy array bit for bit (NaN payloads and the sign of zero included)."""
    t, a = t.cpu(), torch.from_numpy(np.ascontiguousarray(a))
    if t.dtype != a.dtype or t.shape != a.shape:
        return False
    if t.is_floating_point():
        it = torch.int32 if t.dtype == torch.float32 else torch.int64
        t, a = t.view(it), a.view(it)
    return torch.equal(t, a)


def assert_same(buf, ref):
    for name in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts"):
        assert same_bits(getattr(buf, name), getattr(ref, name)), name
    assert buf.pos == ref.pos and buf.full == ref.full and buf.size() == ref.size()


@pytest.mark.parametrize("kind", list(ENVS))
def test_matches_sb3_bit_for_bit(kind):
    """7 slots over 23 adds (wraps), episodes of 3-5 steps (auto-resets fire), n not a multiple of 32 (nor of the add
    kernel's 128-environment blocks), timeouts as a mask and as info dicts, one masked reset; every array after every add."""
    make, scale = ENVS[kind]
    n, slots, adds = 300, 7, 23
    env = make(n)
    buf = ReplayBuffer(slots * n + 5, env, seed=1)
    ref = Sb3ReplayBuffer(slots * n + 5, env.lenObs, env.lenAction, n, np.float32 if env.dtype == torch.float32 else np.float64)
    assert buf.buffer_size == ref.buffer_size == slots
    rng = np.random.default_rng(11)
    env.reset()
    buf.on_reset(env)
    last = host_fm(env._obs, n)
    n_done = n_timeout = n_subst = 0
    for k in range(adds):
        if k == 12:   # an explicit masked reset between steps: SB3's _last_obs is what the env now shows
            env.reset(mask=torch.as_tensor(rng.uniform(size=n) < 0.3, device=DEV))
            buf.on_reset(env)
            last = host_fm(env._obs, n)
        env.set_actions(torch.as_tensor(rng.uniform(-scale, scale, (n, env.lenAction)), dtype=env.dtype, device=DEV))
        env.step_async()
        tmask = rng.uniform(size=n) < 0.25
        infos = [{} for _ in range(n)]
        if k % 3 == 0:
            timeouts = None
        elif k % 3 == 1:
            timeouts = torch.as_tensor(tmask, device=DEV)
        else:
            timeouts = [({"TimeLimit.truncated": True} if t else {}) for t in tmask]
        if timeouts is not None:
            for i in np.nonzero(tmask)[0]:
                infos[i]["TimeLimit.truncated"] = True
        buf.add(env, timeouts=timeouts)
        new_obs, done = host_fm(env._obs, n), env._done[:n].cpu().numpy()
        if env.auto_reset:
            term = host_fm(env._terminal_obs, n)
            for i in np.nonzero(done)[0]:
                infos[i]["terminal_observation"] = term[i]
            n_subst += int((term[done != 0] != new_obs[done != 0]).any(axis=1).sum())
        last = store_transition(ref, last, new_obs, host_fm(env._action, n), env._reward[:n].cpu().numpy(), done, infos)
        n_done += int(done.sum())
        n_timeout += int(sum("TimeLimit.truncated" in i for i in infos))
        assert_same(buf, ref)
    assert same_bits(buf.last_obs[:, :n], last.T)
    assert n_done > n and n_timeout > 0 and ref.full
    assert n_subst > 0 or not env.auto_reset   # the terminal observation differed from the reset one


def filled_buffer(slots=7, n=300, dtype=torch.float64, seed=0):
    """A buffer whose every stored value is distinct (rows identify their slot and environment)."""
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", dtype=dtype, device=DEV, seed=1)
    buf = ReplayBuffer(slots * n, env, seed=seed)
    g = torch.Generator(device=DEV).manual_seed(5)
    m = slots * n
    buf.observations.copy_(torch.arange(m * 9, dtype=dtype, device=DEV).reshape(slots, n, 9))
    buf.next_observations.copy_(-1 - torch.arange(m * 9, dtype=dtype, device=DEV).reshape(slots, n, 9))
    buf.actions.copy_(1e6 + torch.arange(m * 8, dtype=dtype, device=DEV).reshape(slots, n, 8))
    buf.rewards.copy_(0.5 + torch.arange(m, dtype=dtype, device=DEV).reshape(slots, n))
    buf.dones.copy_(torch.randint(0, 2, (slots, n), generator=g, device=DEV, dtype=torch.uint8))
    buf.timeouts.copy_(torch.randint(0, 2, (slots, n), generator=g, device=DEV, dtype=torch.uint8))
    return env, buf


def set_cursor(buf, pos, adds, calls, seed=None):
    d = buf.state_dict()
    d["cursor"] = torch.tensor([pos, adds, calls, pos << 32, 0], dtype=torch.int64)
    if seed is not None:
        d["seed"] = seed
    buf.load_state_dict(d)


@pytest.mark.parametrize("pos,adds,calls,seed", [(3, 3, 0, 123), (5, 12, 2 ** 32 + 5, 2 ** 63 + 12345), (0, 7, 17, 2 ** 64 - 1)],
                         ids=["partly_filled", "wrapped_call_above_2^32_seed_above_2^63", "just_full"])
def test_sampler_against_numpy_philox(pos, adds, calls, seed):
    slots, n, B = 7, 300, 5000
    _, buf = filled_buffer(slots, n)
    set_cursor(buf, pos, adds, calls, seed)
    size = slots if adds >= slots else pos
    for c in (calls, calls + 1):
        out = buf.sample(B)
        slot, env = replay_sample_indices(seed, c, B, size, n)
        assert slot.max() < size and (size == slots or slot.max() == size - 1)
        s, e = torch.as_tensor(slot, device=DEV), torch.as_tensor(env, device=DEV)
        assert torch.equal(out.observations, buf.observations[s, e]) and torch.equal(out.next_observations, buf.next_observations[s, e])
        assert torch.equal(out.actions, buf.actions[s, e]) and torch.equal(out.rewards, buf.rewards[s, e][:, None])
        want = buf.dones[s, e].double() * (1 - buf.timeouts[s, e].double())
        assert torch.equal(out.dones, want[:, None]) and out.dones.shape == (B, 1)
        assert 0 < float(out.dones.sum()) < float(buf.dones[s, e].double().sum())
    assert buf.cursor.tolist() == [pos, adds, calls + 2, pos << 32, 0]


def test_uniformity_chi_square():
    from scipy import stats
    slots, n, B = 37, 1000, 2 ** 22
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", dtype=torch.float32, device=DEV)
    buf = ReplayBuffer(slots * n, env, seed=2024)
    buf.observations[..., 0] = torch.arange(slots, dtype=torch.float32, device=DEV)[:, None]
    buf.observations[..., 1] = torch.arange(n, dtype=torch.float32, device=DEV)[None, :]
    set_cursor(buf, 3, slots + 3, 0)
    out = buf.sample(B).observations
    hs = torch.bincount(out[:, 0].long(), minlength=slots).cpu().numpy()
    he = torch.bincount(out[:, 1].long(), minlength=n).cpu().numpy()
    assert hs.sum() == B and len(hs) == slots and len(he) == n
    assert stats.chisquare(hs).pvalue > 1e-3 and stats.chisquare(he).pvalue > 1e-3
    # partly filled: only slots < pos
    set_cursor(buf, 5, 5, 1)
    hs = torch.bincount(buf.sample(B).observations[:, 0].long(), minlength=slots).cpu().numpy()
    assert hs[5:].sum() == 0 and stats.chisquare(hs[:5]).pvalue > 1e-3


def test_graph_replay_equals_eager_twin():
    n, slots, T, R, B = 1000, 7, 8, 3, 512
    mk = lambda: BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, maxSteps=5, seed=9)
    envg, envt = mk(), mk()
    bufg, buft = ReplayBuffer(slots * n, envg, seed=77), ReplayBuffer(slots * n, envt, seed=77)
    pol = SquashedGaussianPolicy(9, 6, device=DEV, seed=1, action_noise_std=0.1)
    for e, b in ((envg, bufg), (envt, buft)):
        e.reset()
        b.on_reset(e)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    outs = []
    with torch.cuda.graph(graph):
        for k in range(T):
            pol.act(envg, step=k)
            envg.step_async()
            bufg.add(envg)
            outs.append(bufg.sample(B))
    replays = []
    for _ in range(R):
        graph.replay()
        torch.cuda.synchronize()
        replays.append([[t.clone() for t in o] for o in outs])
    eager = []
    for k in range(T * R):
        pol.act(envt, step=k % T)
        envt.step_async()
        buft.add(envt)
        eager.append(buft.sample(B))
    for name in ReplayBuffer._STATE:
        assert torch.equal(getattr(bufg, name), getattr(buft, name)), name
    assert bufg.cursor.tolist() == [(T * R) % slots, T * R, T * R, ((T * R) % slots) << 32, 0]
    for r in range(R):
        for k in range(T):
            for a, b in zip(replays[r][k], eager[r * T + k]):
                assert torch.equal(a, b), (r, k)
    assert not torch.equal(replays[0][T - 1][0], replays[1][T - 1][0]) and not torch.equal(replays[1][T - 1][0], replays[2][T - 1][0])


def test_state_dict_round_trip():
    n = 300
    env = BlueROV2Heavy3DoFVecEnv(n, dtype=torch.float32, device=DEV, maxSteps=4, seed=2)
    a = ReplayBuffer(5 * n, env, seed=3)
    env.reset()
    a.on_reset(env)
    rng = np.random.default_rng(1)
    for _ in range(7):
        env.step_async(torch.as_tensor(rng.uniform(-1, 1, (n, 3)), dtype=torch.float32, device=DEV))
        a.add(env)
        a.sample(16)
    b = ReplayBuffer(5 * n, env, seed=99)
    b.load_state_dict(a.state_dict())
    assert b.seed == 3 and b.pos == a.pos and b.full and b.size() == 5
    env.step_async(torch.as_tensor(rng.uniform(-1, 1, (n, 3)), dtype=torch.float32, device=DEV))
    a.add(env, timeouts=torch.ones(n, dtype=torch.bool, device=DEV))
    b.add(env, timeouts=torch.ones(n, dtype=torch.bool, device=DEV))
    for name in ReplayBuffer._STATE:
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    for x, y in zip(a.sample(1000), b.sample(1000)):
        assert torch.equal(x, y)


def test_benchmark_size_first_and_last_slot_after_wrap():
    """131 072 environments of the 6DoF env, 2^23 transitions (64 slots), 66 adds: slots 0 and 63 against the restatement."""
    n, size, adds = 131072, 2 ** 23, 66
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, maxSteps=3, seed=12)
    buf = ReplayBuffer(size, env, seed=5)
    ref = Sb3ReplayBuffer(size, 9, 6, n, np.float32)
    assert buf.buffer_size == 64
    g = torch.Generator(device=DEV).manual_seed(3)
    env.reset()
    buf.on_reset(env)
    last = host_fm(env._obs, n)
    for k in range(adds):
        env.set_actions(torch.rand((6, n), generator=g, device=DEV) * 2 - 1)
        env.step_async()
        tmask = torch.rand(n, generator=g, device=DEV) < 0.1
        buf.add(env, timeouts=tmask)
        done, tm = env._done[:n].cpu().numpy(), tmask.cpu().numpy()
        term = host_fm(env._terminal_obs, n)
        infos = [{} for _ in range(n)]
        for i in np.nonzero(done)[0]:
            infos[i]["terminal_observation"] = term[i]
        for i in np.nonzero(tm)[0]:
            infos[i]["TimeLimit.truncated"] = True
        last = store_transition(ref, last, host_fm(env._obs, n), host_fm(env._action, n), env._reward[:n].cpu().numpy(), done, infos)
    assert buf.pos == ref.pos == 2 and buf.full and buf.size() == 64
    for s in (0, 63):
        for name in ("observations", "next_observations", "actions", "rewards", "dones", "timeouts"):
            assert same_bits(getattr(buf, name)[s], getattr(ref, name)[s]), (s, name)


def test_errors():
    n = 300
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", dtype=torch.float32, device=DEV, maxSteps=3)
    buf = ReplayBuffer(4 * n, env)
    with pytest.raises(ValueError, match="empty"):
        buf.sample(8)
    for bad in (BlueROV2Heavy6DoFVecEnv(n + 1, action_mode="rpm", device=DEV), BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", dtype=torch.float64, device=DEV),
                BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", device=DEV)):
        with pytest.raises(ValueError, match="does not match"):
            buf.add(bad)
    no_term = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", device=DEV, record_terminal_obs=False)
    with pytest.raises(ValueError, match="terminal"):
        ReplayBuffer(4 * n, no_term).add(no_term)
    with pytest.raises(ValueError, match="buffer_size"):
        ReplayBuffer(0, env)
    env.reset()
    buf.on_reset(env)
    with pytest.raises(ValueError, match="timeouts"):
        buf.add(env, timeouts=torch.zeros(n - 1, dtype=torch.bool, device=DEV))
    with pytest.raises(ValueError, match="timeouts"):
        buf.add(env, timeouts=[{}] * (n - 1))
    with pytest.raises(ValueError, match="timeouts"):
        buf.add(env, timeouts=torch.zeros(n + 1, dtype=torch.bool, device=DEV))
    for bad in ([5, 5, 0, 5 << 32, 0], [1, 1, 0, 0, 0], [2, 1, 0, 2 << 32, 0], [1, 1, 0, (1 << 32) + 3, 0], [1, 1, 0, 1 << 32, 2]):
        d = buf.state_dict()
        d["cursor"] = torch.tensor(bad, dtype=torch.int64)
        with pytest.raises(ValueError, match="cursor"):
            buf.load_state_dict(d)
    buf.add(env)
    for b in (0, -1, 2 ** 31):
        with pytest.raises(ValueError, match="batch_size"):
            buf.sample(b)
    assert buf.sample(1).observations.shape == (1, 9)
    # the C entries: null pointers, obs_dim above MVRL_REPLAY_MAX_DIM
    lib = _lib.load()
    st = lambda **kw: _lib.MvrlReplayStorage(**dict({f: getattr(buf._storage, f) for f, _ in _lib.MvrlReplayStorage._fields_}, **kw))
    stream = _lib.current_stream(env.device)
    add = lambda s, obs_dim=9, obs=env._obs: lib.mvrl_replay_add(0, n, env.ld, obs_dim, 8, buf.buffer_size, C.byref(s), _lib.ptr(obs),
                                                                 _lib.ptr(env._terminal_obs), _lib.ptr(env._action), _lib.ptr(env._reward),
                                                                 _lib.ptr(env._done), None, stream)
    out = [torch.empty(64, dtype=torch.float32, device=DEV) for _ in range(5)]
    sample = lambda s, obs_dim=9: lib.mvrl_replay_sample(0, n, obs_dim, 8, buf.buffer_size, C.byref(s), 4, 0, *[_lib.ptr(t) for t in out], stream)
    assert add(st(observations=None)) == -1 and b"null" in lib.mvrl_last_error()
    assert add(st(cursor=None)) == -1 and sample(st(timeouts=None)) == -1
    assert add(st(), obs=None) == -1
    assert add(st(), obs_dim=17) == -1 and b"obs_dim" in lib.mvrl_last_error()
    assert sample(st(), obs_dim=17) == -1
    host = np.zeros(9 * env.ld, dtype=np.float32)   # host memory in the slots MVRL_ON_DEVICE_OF treats as inputs
    assert lib.mvrl_replay_add(0, n, env.ld, 9, 8, buf.buffer_size, C.byref(st()), C.c_void_p(host.ctypes.data), None,
                               _lib.ptr(env._action), _lib.ptr(env._reward), _lib.ptr(env._done), None, stream) == -1
    assert sample(st(observations=host.ctypes.data)) == -1 and b"device" in lib.mvrl_last_error()
    assert lib.mvrl_replay_sample(0, n, 9, 8, buf.buffer_size, C.byref(st()), 4, 0, None, *[_lib.ptr(t) for t in out[1:]], stream) == -1
    assert add(st()) == 0 and sample(st()) == 0
    torch.cuda.synchronize()
    assert buf.cursor.tolist()[:3] == [2, 2, 2]


def test_pointers_on_two_devices_are_refused():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs a second GPU")
    n = 64
    env = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", device="cuda:0")
    other = BlueROV2Heavy6DoFVecEnv(n, action_mode="rpm", device="cuda:1")
    buf = ReplayBuffer(4 * n, env)
    lib = _lib.load()
    rc = lib.mvrl_replay_add(0, n, env.ld, 9, 8, buf.buffer_size, C.byref(buf._storage), _lib.ptr(other._obs), None,
                             _lib.ptr(env._action), _lib.ptr(env._reward), _lib.ptr(env._done), None, _lib.current_stream(env.device))
    assert rc == -1 and b"device" in lib.mvrl_last_error()
    rc = lib.mvrl_replay_add(0, n, env.ld, 9, 8, buf.buffer_size, C.byref(buf._storage), _lib.ptr(env._obs), None,
                             _lib.ptr(other._action), _lib.ptr(env._reward), _lib.ptr(env._done), None, _lib.current_stream(env.device))
    assert rc == -1
