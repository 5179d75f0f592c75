"""CPU: the host side of ``Critic`` (marinevehiclereinforcementlearning_b200/policy.py) - the parameters it keeps are the
learner's own tensors (a module's ``named_parameters()`` or a mapping, ``critic.`` prefix stripped), while ``CriticTarget``'s
parsing still detaches - and the C entries' refusals that need no device."""
import ctypes as C
import os

import pytest
import torch

from marinevehiclereinforcementlearning_b200 import _lib
from marinevehiclereinforcementlearning_b200 import policy as P


class SB3Critic(torch.nn.Module):
    def __init__(self, obs_dim, act_dim, n_critics, n_out):
        super().__init__()
        for i in range(n_critics):
            self.add_module("qf%d" % i, torch.nn.Sequential(
                torch.nn.Linear(obs_dim + act_dim, 128), torch.nn.GELU(), torch.nn.Linear(128, 128), torch.nn.GELU(),
                torch.nn.Linear(128, 128), torch.nn.GELU(), torch.nn.Linear(128, n_out)))


class Policy(torch.nn.Module):
    """A SAC / TQC policy's layout: critic and critic_target side by side."""

    def __init__(self):
        super().__init__()
        self.critic = SB3Critic(9, 6, 2, 25)
        self.critic_target = SB3Critic(9, 6, 2, 25)


def test_undetached_tensors_are_the_parameters():
    m = SB3Critic(9, 6, 2, 25)
    got = P._critic_tensors(dict(m.named_parameters()), 9, 6, 2, 25, prefixes=("critic.",), detach=False)
    own = dict(m.named_parameters())
    assert list(got) == list(P.critic_param_shapes(9, 6, 2, 25))
    for k, t in got.items():
        assert t is own[k] and t.requires_grad


def test_policy_module_gives_the_online_critic():
    pol = Policy()
    got = P._critic_tensors(dict(pol.named_parameters()), 9, 6, 2, 25, prefixes=("critic.",), detach=False)
    for k, t in got.items():
        assert t is dict(pol.critic.named_parameters())[k]


def test_critic_target_parsing_still_detaches():
    pol = Policy()
    got = P._critic_tensors(dict(pol.named_parameters()), 9, 6, 2, 25)
    for k, t in got.items():
        src = dict(pol.critic_target.named_parameters())[k]
        assert not t.requires_grad and t.data_ptr() == src.data_ptr()


def test_undetached_parsing_keeps_the_checks():
    m = SB3Critic(9, 6, 2, 25)
    sd = dict(m.named_parameters())
    with pytest.raises(ValueError, match="expected the 3 critics"):
        P._critic_tensors(sd, 9, 6, 3, 25, prefixes=("critic.",), detach=False)
    with pytest.raises(ValueError, match="has shape"):
        P._critic_tensors(sd, 9, 6, 2, 24, prefixes=("critic.",), detach=False)


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def test_c_entries_refuse_a_null_handle(lib):
    assert lib.mvrl_critic_saved_bytes(None, 128) == 0
    assert lib.mvrl_critic_grad_scratch(None, 128) == 0
    assert lib.mvrl_critic_forward(None, 1, None, None, None, None, None) == -1
    assert "null handle" in lib.mvrl_last_error().decode()
    assert lib.mvrl_critic_backward(None, 1, None, None, None, None, None, None, None, None) == -1
    assert "null handle" in lib.mvrl_last_error().decode()
