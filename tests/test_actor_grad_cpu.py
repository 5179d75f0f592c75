"""CPU: the host side of ``Actor`` (marinevehiclereinforcementlearning_b200/policy.py) - the parameters it keeps are the
learner's own tensors (a module's ``named_parameters()``, a policy module's ``actor.*`` entries, or a mapping), the
refusals that need no device, the C entries' refusals of a null handle - and the NumPy restatement of its Gaussian draws
(Philox4x32-10 stream 11), which tests/test_actor_grad_gpu.py compares the kernel's ``eps`` with."""
import os

import numpy as np
import pytest
import torch

from marinevehiclereinforcementlearning_b200 import _lib
from marinevehiclereinforcementlearning_b200 import policy as P
from oracle import oracle_np as o

STREAM = 11


def stream11_pair(seed, rows, call, pr):
    """Pair ``pr`` (action dimensions 2 pr, 2 pr + 1) of ``Actor.action_log_prob``'s standard normals of ``rows`` at device
    call number ``call``: Philox4x32-10 with counter (row, call lo, call hi, 11 * 65536 + pr) and key (seed lo, seed hi),
    Box-Muller on the 24-bit words as the actor's draws.  Returns (k1, k2, z0, z1) like ``oracle_np.philox_normal_pair``."""
    rows = np.atleast_1d(np.asarray(rows, dtype=np.uint64))
    ctr = np.stack([rows & np.uint64(0xFFFFFFFF), np.full(rows.shape, call & 0xFFFFFFFF, dtype=np.uint64),
                    np.full(rows.shape, (call >> 32) & 0xFFFFFFFF, dtype=np.uint64),
                    np.full(rows.shape, STREAM * 65536 + pr, dtype=np.uint64)], axis=1).astype(np.uint32)
    w = o.philox4x32(ctr, (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF))
    k1, k2 = w[:, 0] >> np.uint32(8), w[:, 1] >> np.uint32(8)
    r = np.sqrt(-2.0 * np.log(o.normal_pair_u1(k1).astype(np.float64)))
    theta = o.TWO_PI * (k2.astype(np.float64) * (1.0 / 16777216.0))
    return k1, k2, r * np.cos(theta), r * np.sin(theta)


class SB3Actor(torch.nn.Module):
    """SB3's SAC / TQC ``Actor`` parameter layout (no gSDE): latent_pi = Sequential(Linear, GELU, Linear, GELU, Linear, GELU)."""

    def __init__(self, obs_dim, act_dim):
        super().__init__()
        self.latent_pi = torch.nn.Sequential(torch.nn.Linear(obs_dim, 128), torch.nn.GELU(), torch.nn.Linear(128, 128), torch.nn.GELU(),
                                             torch.nn.Linear(128, 128), torch.nn.GELU())
        self.mu = torch.nn.Linear(128, act_dim)
        self.log_std = torch.nn.Linear(128, act_dim)


class Policy(torch.nn.Module):
    """A SAC policy's layout: actor, critic and critic_target side by side."""

    def __init__(self):
        super().__init__()
        self.actor = SB3Actor(9, 6)
        self.critic = torch.nn.Linear(15, 1)
        self.critic_target = torch.nn.Linear(15, 1)


def test_stream11_counter_layout():
    """The kernel draws stream 11 through the actor's normal_pair with env id = row | call lo << 32 and step = call hi:
    the restatement equals ``philox_normal_pair`` keyed that way, word for word, at calls on both sides of 2^32; the call
    number, the row, the pair and both seed words each change the draws, and stream 11 is not the critic target's 10."""
    seed = 0xD1B54A32D192ED03
    rows = np.arange(0, 5000, dtype=np.uint64)
    for call in (0, 1, 2 ** 32 - 1, 2 ** 32 + 5, 2 ** 40 + 3):
        for pr in range(4):
            k1, k2, z0, z1 = stream11_pair(seed, rows, call, pr)
            env = rows | np.uint64((call & 0xFFFFFFFF) << 32)
            q1, q2, y0, y1 = o.philox_normal_pair(seed, env, call >> 32, pr, STREAM)
            assert np.array_equal(k1, q1) and np.array_equal(k2, q2) and np.array_equal(z0, y0) and np.array_equal(z1, y1)
    base = stream11_pair(seed, rows, 7, 0)[0]
    for other in (stream11_pair(seed, rows, 8, 0)[0], stream11_pair(seed, rows, 7 + 2 ** 32, 0)[0], stream11_pair(seed, rows, 7, 1)[0],
                  stream11_pair(seed & 0xFFFFFFFF, rows, 7, 0)[0], stream11_pair(seed, rows + np.uint64(1), 7, 0)[0],
                  o.philox_normal_pair(seed, rows | np.uint64(7 << 32), 0, 0, 10)[0]):
        assert np.mean(other == base) < 0.01
    z = np.concatenate([stream11_pair(seed, np.arange(2 ** 18, dtype=np.uint64), 3, pr)[2] for pr in range(4)])
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01


def test_module_policy_and_mapping_give_the_parameters():
    m = SB3Actor(9, 6)
    own = dict(m.named_parameters())
    for named in (own, {"actor." + k: v for k, v in own.items()}):
        got = P._actor_tensors(named, 9, 6, detach=False)
        assert list(got) == list(P.squashed_param_shapes(9, 6))
        for k, t in got.items():
            assert t is own[k] and t.requires_grad
    pol = Policy()
    got = P._actor_tensors(dict(pol.named_parameters()), 9, 6, detach=False)
    for k, t in got.items():
        assert t is dict(pol.actor.named_parameters())[k]
    # the default still detaches (SquashedGaussianPolicy.load_state_dict)
    for k, t in P._actor_tensors(own, 9, 6).items():
        assert not t.requires_grad and t.data_ptr() == own[k].data_ptr()


def test_refusals_without_a_device():
    m = SB3Actor(9, 6)
    for obs_dim, act_dim in ((17, 6), (9, 9), (0, 6), (9, 0)):
        with pytest.raises(ValueError, match="obs_dim <= 16 and 1 <= act_dim <= 8"):
            P.Actor(m, obs_dim, act_dim)
    with pytest.raises(ValueError, match="CUDA device"):
        P.Actor(m, 9, 6)
    sd = dict(m.named_parameters())
    with pytest.raises(ValueError, match="gSDE"):
        P.Actor(dict(sd, log_std=torch.zeros(6)), 9, 6)
    with pytest.raises(ValueError, match="no 'mu.bias'"):
        P.Actor({k: v for k, v in sd.items() if k != "mu.bias"}, 9, 6)
    with pytest.raises(ValueError, match="has shape"):
        P.Actor(sd, 9, 5)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def test_c_entries_refuse_a_null_handle(lib):
    assert lib.mvrl_actor_saved_bytes(None, 128) == 0
    assert lib.mvrl_actor_grad_scratch(None, 128) == 0
    assert lib.mvrl_actor_forward(None, 1, None, None, None, None, None, 0, None, None) == -1
    assert "null handle" in lib.mvrl_last_error().decode()
    assert lib.mvrl_actor_backward(None, 1, None, None, None, None, None, None, None) == -1
    assert "null handle" in lib.mvrl_last_error().decode()
