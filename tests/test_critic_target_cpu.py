"""CPU: the host side of ``CriticTarget`` (marinevehiclereinforcementlearning_b200/policy.py) - parsing of SB3 critic state
dicts in their three forms, the configuration and constructor refusals - and the NumPy restatement of the critic target's
Gaussian draws (Philox4x32-10 stream 10), which tests/test_critic_target_gpu.py compares the kernel's ``eps`` with."""
import numpy as np
import pytest
import torch

from marinevehiclereinforcementlearning_b200 import policy as P
from oracle import oracle_np as o

STREAM = 10


def stream10_pair(seed, rows, call, pr):
    """Pair ``pr`` (action dimensions 2 pr, 2 pr + 1) of the critic target's standard normals of sampled ``rows`` at device
    call number ``call``: Philox4x32-10 with counter (row, call lo, call hi, 10 * 65536 + pr) and key (seed lo, seed hi),
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


def critic_state_dict(obs_dim, act_dim, n_critics, n_out, seed=0, prefix=""):
    g = torch.Generator().manual_seed(seed)
    return {prefix + k: torch.randn(s, generator=g) for k, s in P.critic_param_shapes(obs_dim, act_dim, n_critics, n_out).items()}


def test_stream10_counter_layout():
    """The kernel draws stream 10 through the actor's normal_pair with env id = row | call lo << 32 and step = call hi:
    the restatement equals ``philox_normal_pair`` keyed that way, word for word, at calls on both sides of 2^32; the call
    number, the row, the pair and both seed words each change the draws."""
    seed = 0xD1B54A32D192ED03
    rows = np.arange(0, 5000, dtype=np.uint64)
    for call in (0, 1, 2 ** 32 - 1, 2 ** 32 + 5, 2 ** 40 + 3):
        for pr in range(4):
            k1, k2, z0, z1 = stream10_pair(seed, rows, call, pr)
            env = rows | np.uint64((call & 0xFFFFFFFF) << 32)
            q1, q2, y0, y1 = o.philox_normal_pair(seed, env, call >> 32, pr, STREAM)
            assert np.array_equal(k1, q1) and np.array_equal(k2, q2) and np.array_equal(z0, y0) and np.array_equal(z1, y1)
    base = stream10_pair(seed, rows, 7, 0)[0]
    for other in (stream10_pair(seed, rows, 8, 0)[0], stream10_pair(seed, rows, 7 + 2 ** 32, 0)[0], stream10_pair(seed, rows, 7, 1)[0],
                  stream10_pair(seed & 0xFFFFFFFF, rows, 7, 0)[0], stream10_pair(seed, rows + np.uint64(1), 7, 0)[0],
                  o.philox_normal_pair(seed, rows | np.uint64(7 << 32), 0, 0, 9)[0]):
        assert np.mean(other == base) < 0.01
    z = np.concatenate([stream10_pair(seed, np.arange(2 ** 18, dtype=np.uint64), 3, pr)[2] for pr in range(4)])
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01


@pytest.mark.parametrize("form", ["module", "critic", "critic_target"])
def test_state_dict_forms(form):
    """A critic module state dict, a policy state dict with critic.* only, and one with both (critic_target.* taken)."""
    target = critic_state_dict(9, 6, 2, 25, seed=1)
    online = critic_state_dict(9, 6, 2, 25, seed=2)
    if form == "module":
        sd, want = target, target
    elif form == "critic":
        sd, want = {"critic." + k: v for k, v in online.items()}, online
    else:
        sd = {"critic." + k: v for k, v in online.items()}
        sd.update({"critic_target." + k: v for k, v in target.items()})
        sd["actor.latent_pi.0.weight"] = torch.zeros(128, 9)
        want = target
    got = P._critic_tensors(sd, 9, 6, 2, 25)
    assert list(got) == list(P.critic_param_shapes(9, 6, 2, 25))
    for k, t in got.items():
        assert t.data_ptr() == want[k].data_ptr()   # references, not copies (share=True keeps them)
    assert tuple(got["qf0.0.weight"].shape) == (128, 15) and tuple(got["qf1.6.weight"].shape) == (25, 128)


def test_state_dict_refusals():
    sd = critic_state_dict(9, 6, 2, 25)
    for bad, match in (({k: v for k, v in sd.items() if k != "qf1.4.bias"}, "no 'qf1.4.bias'"),
                       (dict(sd, **{"qf0.2.weight": torch.zeros(64, 128)}), "shape"),
                       (dict(sd, **{"qf0.6.weight": torch.zeros(1, 128), "qf0.6.bias": torch.zeros(1)}), "shape"),
                       (dict(sd, **{"qf0.8.weight": torch.zeros(25, 25), "qf0.8.bias": torch.zeros(25)}), "beyond"),
                       (critic_state_dict(9, 6, 3, 25), "critics"),
                       (critic_state_dict(9, 6, 1, 25), "critics"),
                       ({}, "critics")):
        with pytest.raises(ValueError, match=match):
            P._critic_tensors(bad, 9, 6, 2, 25)
    # SAC: one output per critic
    P._critic_tensors(critic_state_dict(11, 3, 2, 1), 11, 3, 2, 1)
    with pytest.raises(ValueError, match="shape"):
        P._critic_tensors(critic_state_dict(11, 3, 2, 25), 11, 3, 2, 1)


def test_config_and_constructor_refusals():
    assert P.critic_target_config("tqc", 2, 25, 2, 9, 6) == (25, 2, 46)
    assert P.critic_target_config("tqc", 5, 32, 31, 1, 1) == (32, 31, 5)
    assert P.critic_target_config("sac", 2, 25, 2, 11, 3) == (1, 0, 1)
    for args, match in ((("td3", 2, 25, 2, 9, 6), "kind"), (("tqc", 0, 25, 2, 9, 6), "n_critics"), (("tqc", 6, 25, 2, 9, 6), "n_critics"),
                        (("tqc", 2, 0, 0, 9, 6), "n_quantiles"), (("tqc", 2, 33, 2, 9, 6), "n_quantiles"),
                        (("tqc", 2, 25, 25, 9, 6), "keep"), (("tqc", 2, 25, -1, 9, 6), "keep"), (("sac", 2, 1, 0, 11, 6), "16"),
                        (("tqc", 2, 25, 2, 11, 6), "16")):   # obs_dim + act_dim > 16: refused before any state dict is read
        with pytest.raises(ValueError, match=match):
            P.critic_target_config(*args)
    # the actor: a SquashedGaussianPolicy with precision="fp32" (checked before any device work)
    for actor in (None, object(), "fp32"):
        with pytest.raises(ValueError, match="SquashedGaussianPolicy"):
            P.CriticTarget(actor)
    bf16 = object.__new__(P.SquashedGaussianPolicy)
    bf16.precision = "bf16"
    with pytest.raises(ValueError, match="fp32"):
        P.CriticTarget(bf16)
    fp32 = object.__new__(P.SquashedGaussianPolicy)
    fp32.precision, fp32.obs_dim, fp32.act_dim, fp32.device = "fp32", 11, 6, torch.device("cuda", 0)
    with pytest.raises(ValueError, match="16"):
        P.CriticTarget(fp32)
    fp32.obs_dim = 9
    with pytest.raises(ValueError, match="n_quantiles"):
        P.CriticTarget(fp32, n_quantiles=40)
