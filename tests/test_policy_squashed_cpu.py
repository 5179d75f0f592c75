"""CPU: the SB3 key mapping of SquashedGaussianPolicy, the squashed head's C ABI declarations, and its entry points'
argument checks on an interpreter that sees no CUDA device."""
import os
import re
import subprocess
import sys
import textwrap

import pytest
import torch

from conftest import ROOT
from marinevehiclereinforcementlearning_b200 import _lib
from marinevehiclereinforcementlearning_b200.policy import actor_params_from_state_dict, squashed_param_shapes


def actor_sd(obs_dim=9, act_dim=6):
    g = torch.Generator().manual_seed(0)
    return {k: torch.randn(s, generator=g) for k, s in squashed_param_shapes(obs_dim, act_dim).items()}


def test_actor_state_dict_is_taken_as_is():
    sd = actor_sd()
    got = actor_params_from_state_dict(sd, 9, 6)
    assert set(got) == set(sd) and all(torch.equal(got[k], sd[k]) for k in sd)
    assert all(got[k].dtype == torch.float32 and got[k].data_ptr() != sd[k].data_ptr() for k in sd)   # copies


def test_policy_state_dict_prefix_and_ignored_keys():
    """A whole SAC / TQC policy state dict: the actor.* keys are used, critic / critic_target keys ignored; float64 or numpy
    values are converted."""
    sd = actor_sd(5, 3)
    full = {"actor." + k: v.double().numpy() for k, v in sd.items()}
    full.update({"critic.qf0.0.weight": torch.zeros(128, 8), "critic_target.qf1.4.bias": torch.zeros(1),
                 "mu.weight": torch.zeros(3, 128)})   # an unprefixed key next to actor.* keys is not the actor's
    got = actor_params_from_state_dict(full, 5, 3)
    assert set(got) == set(sd)
    assert all(torch.allclose(got[k], sd[k], atol=1e-7) and got[k].dtype == torch.float32 for k in sd)
    assert not torch.equal(got["mu.weight"], torch.zeros(3, 128))


@pytest.mark.parametrize("drop", ["latent_pi.2.weight", "log_std.bias", "mu.weight"])
def test_missing_key_raises(drop):
    sd = actor_sd()
    del sd[drop]
    with pytest.raises(ValueError, match=re.escape(drop)):
        actor_params_from_state_dict(sd, 9, 6)


def test_shape_mismatch_raises():
    with pytest.raises(ValueError, match="latent_pi.0.weight"):
        actor_params_from_state_dict(actor_sd(9, 6), 11, 6)      # another obs_dim
    sd = actor_sd()
    sd["latent_pi.4.weight"] = torch.zeros(256, 128)               # another net_arch
    with pytest.raises(ValueError, match="latent_pi.4.weight"):
        actor_params_from_state_dict(sd, 9, 6)


def test_gsde_actor_raises():
    """use_sde=True: log_std is a Parameter [latent, act_dim] (key 'log_std'), not a Linear layer."""
    sd = {k: v for k, v in actor_sd().items() if not k.startswith("log_std.")}
    sd["log_std"] = torch.zeros(128, 6)
    with pytest.raises(ValueError, match="gSDE"):
        actor_params_from_state_dict({"actor." + k: v for k, v in sd.items()}, 9, 6)


def test_abi_declares_the_squashed_head():
    header = open(os.path.join(ROOT, "include", "mvrl.h")).read()
    for name in ("mvrl_policy_create_head", "mvrl_policy_set_weights_squashed", "mvrl_policy_act_ex"):
        assert re.search(r"MVRL_API\s+int\s+%s\s*\(" % name, header), name
        assert name in _lib.PROTOTYPES
    assert re.search(r"#define MVRL_POLICY_HEAD_FIXED_STD 0\b", header) and re.search(r"#define MVRL_POLICY_HEAD_SQUASHED 1\b", header)
    assert (_lib.POLICY_HEAD_FIXED_STD, _lib.POLICY_HEAD_SQUASHED) == (0, 1)
    assert len(_lib.PROTOTYPES["mvrl_policy_set_weights_squashed"][1]) == 12
    assert len(_lib.PROTOTYPES["mvrl_policy_act_ex"][1]) == len(_lib.PROTOTYPES["mvrl_policy_act"][1]) + 1


NO_DEVICE = textwrap.dedent("""
    import ctypes as C, sys
    sys.path.insert(0, %r)
    import pytest, torch
    from marinevehiclereinforcementlearning_b200 import _lib, SquashedGaussianPolicy
    assert not torch.cuda.is_available()
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.mvrl_policy_create_head(C.byref(h), 0, 9, 6, 2) == -1 and b"head" in lib.mvrl_last_error()   # unknown head
    assert lib.mvrl_policy_create_head(C.byref(h), 0, 9, 6, -1) == -1
    assert lib.mvrl_policy_create_head(C.byref(h), 0, 9, 6, 1) == -3                                     # MVRL_ENODEV
    assert lib.mvrl_policy_create_head(C.byref(h), 0, 9, 9, 1) == -1                                     # act_dim > 8
    w = (C.c_float * 16384)()
    p = C.cast(w, C.c_void_p)
    assert lib.mvrl_policy_set_weights_squashed(None, *([p] * 10), None) == -1
    assert lib.mvrl_policy_set_weights_squashed(None, *([p] * 10), p) == -1
    assert lib.mvrl_policy_act_ex(None, 1, 32, p, p, None, None, p, None, 0, 0, 0, 0, None) == -1
    with pytest.raises(RuntimeError):
        SquashedGaussianPolicy(9, 6)
    print("squashed head no device ok")
""")


def test_entry_points_without_a_device():
    """In a fresh interpreter that sees no device (CUDA_VISIBLE_DEVICES=""): an unknown head is MVRL_EINVAL, a valid one
    MVRL_ENODEV, calls without a handle MVRL_EINVAL, and the Python class refuses to run."""
    res = subprocess.run([sys.executable, "-c", NO_DEVICE % ROOT], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0 and "squashed head no device ok" in res.stdout, res.stdout[-2000:] + res.stderr[-2000:]
