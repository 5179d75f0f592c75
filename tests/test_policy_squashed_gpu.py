"""GPU: the squashed Gaussian head of the fused rollout actor (the Actor of SB3 SAC / sb3_contrib TQC; csrc/mvrl_policy.cu)
against plain PyTorch restatements of the network and of SB3's SquashedDiagGaussianDistribution."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import (AuvVecEnv, BlueROV2Heavy3DoFVecEnv, BlueROV2Heavy6DoFVecEnv, MlpGaussianPolicy,
                                                         SquashedGaussianPolicy, _lib)

DEV = "cuda"

# Tolerances of mu / log_std (the head layers' outputs; mu before any tanh) against
#  * the bf16-mirroring restatement: the operands are the same bf16 values; what differs is the tanh.approx of the hidden
#    GELUs (2^-11 relative), which now and then flips the bf16 rounding of an activation (one bf16 ulp, 2^-8 relative, of
#    one of 128 terms), and the fp32 summation order - the fixed head's 6e-3 budget (measured here, B200: 2.4e-3 max over
#    every size and shape below);
#  * the fp32 / erf-GELU network SB3 evaluates: bf16 operands (2^-9 relative per operand over three hidden layers and the
#    head, sums of 128 terms of random sign) + the tanh form of GELU (within 1e-3): measured 4.4e-3 max, bound 1.5e-2.
# Unlike the fixed head's mean these are not compressed by a tanh (slope 1 near the origin, so the same scale).
TOL_BF16, TOL_FP32 = 6e-3, 1.5e-2


def sb3_actor_state_dict(obs_dim, act_dim, seed=3, log_std_bias=(-1.5, -0.3)):
    """A random SB3-named Actor state dict with non-zero biases (nn.Linear layout, fp32)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, fan_in, fan_out in (("latent_pi.0", obs_dim, 128), ("latent_pi.2", 128, 128), ("latent_pi.4", 128, 128),
                                  ("mu", 128, act_dim), ("log_std", 128, act_dim)):
        sd[name + ".weight"] = torch.randn(fan_out, fan_in, generator=g) / math.sqrt(fan_in)
        sd[name + ".bias"] = torch.rand(fan_out, generator=g) * 0.6 - 0.3
    lo, hi = log_std_bias
    sd["log_std.bias"] = torch.rand(act_dim, generator=g) * (hi - lo) + lo
    return sd


def reference_forward(sd, obs_nk, round_bf16=True):
    """Plain PyTorch restatement of the network (the test's reference; the product has no PyTorch path): (mu, clamped
    log_std) [N, act_dim].  ``round_bf16=True`` mirrors the kernel's arithmetic (bf16 operands, tanh-form GELU); ``False``
    is the Actor as SB3 evaluates it: fp32 with ``torch.nn.GELU()`` (the erf form)."""
    r = (lambda t: t.to(torch.bfloat16).to(torch.float32)) if round_bf16 else (lambda t: t)
    approx = "tanh" if round_bf16 else "none"
    p = {k: v.to(obs_nk.device, torch.float32) for k, v in sd.items()}
    h = r(obs_nk.to(torch.float32))
    for i in (0, 2, 4):
        h = r(torch.nn.functional.gelu(h @ r(p["latent_pi.%d.weight" % i]).T + p["latent_pi.%d.bias" % i], approximate=approx))
    mu = h @ r(p["mu.weight"]).T + p["mu.bias"]
    log_std = (h @ r(p["log_std.weight"]).T + p["log_std.bias"]).clamp(-20.0, 2.0)
    return mu, log_std


def make_policy(obs_dim, act_dim, sd, noise=None, seed=3):
    pol = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, seed=seed, action_noise_std=noise)
    pol.load_state_dict(sd)
    return pol


def buffers(obs_dim, act_dim, n, seed=0):
    ld = (n + 31) // 32 * 32
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.zeros((obs_dim, ld), device=DEV)
    obs[:, :n] = torch.rand((obs_dim, n), generator=g, device=DEV) * 2 - 1
    z = lambda k: torch.full((k, ld), 7.0, device=DEV)
    return dict(obs=obs, act=z(act_dim), mean=z(act_dim), log_std=z(act_dim), eps=z(act_dim), logp=torch.full((ld,), 7.0, device=DEV))


def run(pol, b, n, env_id0=11, step=4, deterministic=False):
    pol.act_into(b["obs"], b["act"], n, logp=b["logp"], mean=b["mean"], eps=b["eps"], log_std=b["log_std"], env_id0=env_id0, step=step,
                 deterministic=deterministic)
    torch.cuda.synchronize()
    return b


def head_reference(mu, log_std, eps, act):
    """SB3's squashed sample and log-prob in fp64 from the kernel's own mu / log_std / eps: (tanh(u), log-prob of act)
    with torch.distributions.Normal for the Gaussian part and the tanh Jacobian log(1 - act^2 + 1e-6)."""
    mu, log_std, eps, act = (t.double() for t in (mu, log_std, eps, act))
    std = log_std.exp()
    u = mu + std * eps
    lp = torch.distributions.Normal(mu, std).log_prob(u).sum(1) - torch.log(1.0 - act * act + 1e-6).sum(1)
    return torch.tanh(u), lp


SHAPES = [(9, 6), (5, 3), (11, 3), (1, 1), (16, 8)]


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_squashed_actor_matches_pytorch_reference(obs_dim, act_dim):
    """Tests 1 and 2: mu / log_std against both restatements; act and logp by SB3's formulas from the kernel's own outputs;
    nothing written at or beyond row n."""
    sd = sb3_actor_state_dict(obs_dim, act_dim)
    pol = make_policy(obs_dim, act_dim, sd)
    worst = {}
    for n in (1, 37, 128, 5000, 131072):
        b = run(pol, buffers(obs_dim, act_dim, n), n)
        x = b["obs"][:, :n].T
        mu, ls = (b[k][:, :n].T for k in ("mean", "log_std"))
        mu16, ls16 = reference_forward(sd, x, round_bf16=True)
        mu32, ls32 = reference_forward(sd, x, round_bf16=False)
        e_bf16 = max(float((mu - mu16).abs().max()), float((ls - ls16).abs().max()))
        e_fp32 = max(float((mu - mu32).abs().max()), float((ls - ls32).abs().max()))
        assert e_bf16 < TOL_BF16 and e_fp32 < TOL_FP32, (n, e_bf16, e_fp32)
        eps, act, logp = b["eps"][:, :n].T, b["act"][:, :n].T, b["logp"][:n]
        a_ref, lp_ref = head_reference(mu, ls, eps, act)
        e_act = float((act.double() - a_ref).abs().max())
        e_lp = float((logp.double() - lp_ref).abs().max())
        # act: fp32 fma + expf + tanhf (a few ulp of |u|, slope of tanh <= 1); logp per environment: the eps^2 term (eps
        # recovered exactly here), fp32 sums of act_dim terms up to |log(1e-6)| = 13.8 and logf (1 ulp)
        assert e_act < 2e-6, (n, e_act)
        assert e_lp < 1e-5 * act_dim, (n, e_lp)
        assert bool((act.abs() <= 1.0).all())
        for k in ("act", "mean", "log_std", "eps"):
            assert bool((b[k][:, n:] == 7.0).all()), k
        assert bool((b["logp"][n:] == 7.0).all())
        for k, v in (("bf16", e_bf16), ("fp32", e_fp32), ("act", e_act), ("logp", e_lp)):
            worst[k] = max(worst.get(k, 0.0), v)
    print("squashed head (%d, %d): max |mu, log_std - bf16 ref| %.3g, - fp32 ref %.3g; |act - formula| %.3g; |logp - formula| %.3g"
          % (obs_dim, act_dim, worst["bf16"], worst["fp32"], worst["act"], worst["logp"]))


def test_log_std_clamp():
    """Test 3: log_std biases of +-30 give exactly 2 / -20."""
    for bias, want in ((30.0, 2.0), (-30.0, -20.0)):
        sd = sb3_actor_state_dict(9, 6)
        sd["log_std.bias"] = torch.full((6,), bias)
        pol = make_policy(9, 6, sd)
        n = 1000
        b = run(pol, buffers(9, 6, n), n)
        assert bool((b["log_std"][:, :n] == want).all())
        assert bool(torch.isfinite(b["act"][:, :n]).all()) and bool(torch.isfinite(b["logp"][:n]).all())


def test_action_noise():
    """Test 4: noise on / off with the same seed and step: eps bitwise equal; the noise is N(0, 1), uncorrelated with eps;
    clipping gives exactly +-1 as often as the normal law says; deterministic = tanh(mu) without noise."""
    sd = sb3_actor_state_dict(9, 6)
    noise_std = torch.tensor([0.05, 0.1, 0.15, 0.05, 0.1, 2.0])
    off, on = make_policy(9, 6, sd), make_policy(9, 6, sd, noise=noise_std)
    n = 131072
    bo, bn = run(off, buffers(9, 6, n), n), run(on, buffers(9, 6, n), n)
    assert torch.equal(bo["eps"], bn["eps"]) and torch.equal(bo["mean"], bn["mean"]) and torch.equal(bo["logp"], bn["logp"])
    a_off, a_on, eps = bo["act"][:, :n], bn["act"][:, :n], bo["eps"][:, :n]
    assert bool((a_on.abs() <= 1.0).all())
    s = noise_std.to(DEV)[:, None]
    # entries whose noise cannot reach the clip (|xi| <= 5.9 for the 24-bit Box-Muller): selected on a_off only, so that the
    # selection does not depend on the noise
    free = (a_off.abs() + 6.0 * s < 1.0)[:5]
    xi = ((a_on[:5] - a_off[:5]) / s[:5])[free].double()
    assert xi.numel() > 100000
    assert abs(float(xi.mean())) < 0.02 and abs(float(xi.std()) - 1.0) < 0.02
    assert abs(float((xi ** 3).mean())) < 0.08 and abs(float((xi ** 4).mean()) - 3.0) < 0.2
    corr = float(torch.corrcoef(torch.stack([xi, eps[:5][free].double()]))[0, 1])
    assert abs(corr) < 0.02, corr
    # the wide last dimension (noise_std 2): clipped entries are exactly +-1, as often as P(|a + 2 xi| > 1) given a
    a5, o5 = a_off[5].double(), a_on[5]
    nrm = torch.distributions.Normal(0.0, 1.0)
    p_clip = float((nrm.cdf((-1.0 - a5) / 2.0) + 1.0 - nrm.cdf((1.0 - a5) / 2.0)).mean())
    frac = float((o5.abs() == 1.0).double().mean())
    assert p_clip > 0.3 and abs(frac - p_clip) < 0.01, (frac, p_clip)
    # deterministic: tanh(mu), no noise, eps = 0
    bd = run(on, buffers(9, 6, n), n, deterministic=True)
    assert torch.allclose(bd["act"][:, :n], torch.tanh(bd["mean"][:, :n]), atol=1e-6, rtol=0)
    assert bool((bd["eps"][:, :n] == 0.0).all())


def test_sharding_gives_the_same_draws():
    """Test 5: two shards with env_id0 offsets give bitwise the same eps, noise and act as one launch."""
    sd = sb3_actor_state_dict(9, 6)
    pol = make_policy(9, 6, sd, noise=0.3)
    n, lo = 1000, 512
    b = run(pol, buffers(9, 6, n, seed=2), n, env_id0=0, step=7)
    obs2 = b["obs"][:, lo:lo + 512].contiguous()
    act2, eps2, mean2 = torch.zeros_like(obs2[:6]), torch.zeros_like(obs2[:6]), torch.zeros_like(obs2[:6])
    pol.act_into(obs2, act2, n - lo, eps=eps2, mean=mean2, env_id0=lo, step=7)
    torch.cuda.synchronize()
    assert torch.equal(eps2[:, :n - lo], b["eps"][:, lo:n])
    assert torch.equal(mean2[:, :n - lo], b["mean"][:, lo:n])
    assert torch.equal(act2[:, :n - lo], b["act"][:, lo:n])   # the noise, too: same mean, eps and act


@pytest.mark.parametrize("obs_dim,act_dim", [(9, 6), (5, 3), (16, 8), (1, 1)])
def test_tcgen05_and_mma_sync_squashed_kernels_agree(monkeypatch, obs_dim, act_dim):
    """Test 6: the tcgen05 and the mma.sync squashed kernels on the same inputs: identical eps and noise, mu / log_std
    within the fp32 summation-order difference; sizes around the 128-row tile and more tiles than tile groups.  The noise
    is compared through a head with zero weights (mu = b_mu and log_std = b_log_std exactly in both kernels, so act is
    bitwise a function of eps and the noise)."""
    sd = sb3_actor_state_dict(obs_dim, act_dim)
    sd0 = dict(sd, **{"mu.weight": torch.zeros(act_dim, 128), "log_std.weight": torch.zeros(act_dim, 128)})
    pols = {}
    for flag in ("0", "1"):
        monkeypatch.setenv("MVRL_POLICY_MMA_SYNC", flag)
        pols[flag] = (make_policy(obs_dim, act_dim, sd, noise=0.2), make_policy(obs_dim, act_dim, sd0, noise=0.2))
    for n in (1, 127, 129, 1000, 80000):
        out = {f: (run(p, buffers(obs_dim, act_dim, n, seed=1), n, env_id0=5, step=9), run(p0, buffers(obs_dim, act_dim, n, seed=1), n, env_id0=5, step=9))
               for f, (p, p0) in pols.items()}
        (b5, z5), (bs, zs) = out["0"], out["1"]
        assert torch.equal(b5["eps"], bs["eps"])                   # same draws, bit for bit (also the untouched padding)
        for k in ("mean", "log_std"):
            d = (b5[k][:, :n] - bs[k][:, :n]).abs()
            assert float(d.max()) < 2e-3 and float(d.mean()) < 1e-4, (k, n, float(d.max()))
        assert torch.equal(z5["act"], zs["act"])                   # same noise
        # logp: the same terms, summed in another order (a quad butterfly in the mma.sync kernel) for act_dim > 4
        assert torch.allclose(z5["logp"], zs["logp"], rtol=1e-6, atol=1e-6)
        assert bool((b5["act"][:, n:] == 7.0).all()) and bool((b5["logp"][n:] == 7.0).all())


@pytest.mark.parametrize("which", ["rov6", "rov3", "auv"])
def test_closed_loop(which):
    """Test 7: 20 steps of pol.act(env); env.step() on the env's own buffers: state and logp finite, |act| <= 1."""
    n = 4096
    if which == "rov6":
        env = BlueROV2Heavy6DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, maxSteps=8, auto_reset=True, seed=1)
    elif which == "rov3":
        env = BlueROV2Heavy3DoFVecEnv(n, action_mode="setpoint", dtype=torch.float32, device=DEV, maxSteps=8, auto_reset=True, seed=1)
    else:
        from marinevehiclereinforcementlearning_b200.tag_00_Dec2023_simpleControlTurbulence import flowGenerator
        ltm = np.load(os.path.join(ROOT, "tests", "golden", "golden_legacy.npz"))["ltm"]
        flow = flowGenerator.ReconstructedFlow.synthetic(lt_mean=ltm, nt=8, kind="modes", dtype=torch.float32, device=DEV)
        flow.scale(11., 1., 2., translate=(-1.65, -1.1))
        env = AuvVecEnv(n, flow, dtype=torch.float32, maxSteps=8, auto_reset=True, seed=1)
    pol = SquashedGaussianPolicy(env.lenObs, env.lenAction, device=DEV, seed=1, action_noise_std=0.1)
    env.reset()
    logp = torch.empty(env.ld, device=DEV)
    for _ in range(20):
        pol.act(env, logp=logp)
        assert float(env.actions_fm.abs().max()) <= 1.0
        env.step()
        assert bool(torch.isfinite(logp[:n]).all())
    assert bool(torch.isfinite(env.state if which == "auv" else env.systemState).all())


def test_trained_tqc_actor_predict_is_tanh_mu():
    """A whole TQC policy state dict (actor.* and critic.* keys): predict(obs, deterministic=True) = tanh(mu) of that
    network, within the bf16-class tolerance; state_dict() round-trips."""
    actor = sb3_actor_state_dict(9, 6, seed=8)
    g = torch.Generator().manual_seed(1)
    sd = {"actor." + k: v for k, v in actor.items()}
    sd.update({"critic.qf0.0.weight": torch.randn(128, 15, generator=g), "critic.qf0.0.bias": torch.zeros(128),
               "critic_target.qf0.0.weight": torch.randn(128, 15, generator=g)})
    pol = SquashedGaussianPolicy(9, 6, device=DEV, action_noise_std=0.5).load_state_dict(sd)
    assert all(torch.equal(pol.state_dict()[k], v) for k, v in actor.items())
    obs = np.random.default_rng(0).uniform(-1, 1, (300, 9)).astype(np.float32)
    a, _ = pol.predict(obs, deterministic=True)
    mu16, _ = reference_forward(actor, torch.as_tensor(obs), round_bf16=True)
    mu32, _ = reference_forward(actor, torch.as_tensor(obs), round_bf16=False)
    assert a.shape == (300, 6)
    assert np.abs(a - torch.tanh(mu16).numpy()).max() < TOL_BF16 and np.abs(a - torch.tanh(mu32).numpy()).max() < TOL_FP32
    a1, _ = pol.predict(obs[0], deterministic=True)
    assert a1.shape == (6,) and np.array_equal(a1, a[0])
    pol2 = SquashedGaussianPolicy(9, 6, device=DEV).load_state_dict(pol.state_dict())
    assert np.array_equal(pol2.predict(obs, deterministic=True)[0], a)


def test_wrong_kind_calls_are_rejected():
    """MVRL_EINVAL for: the fixed head's weights on a squashed handle and the other way round, a log_std output on a fixed
    handle, an unknown head; the squashed policy rejects a bad noise vector."""
    lib = _lib.load()
    sq = SquashedGaussianPolicy(9, 6, device=DEV)
    fx = MlpGaussianPolicy(9, 6, device=DEV)
    w = torch.zeros(128 * 128)
    p = C.c_void_p(w.data_ptr())
    assert lib.mvrl_policy_set_weights(sq._h, *([p] * 9)) == -1
    assert lib.mvrl_policy_set_weights_squashed(fx._h, *([p] * 10), None) == -1
    b = buffers(9, 6, 64)
    with pytest.raises(RuntimeError):
        fx.act_into(b["obs"], b["act"], 64, log_std=b["log_std"])
    h = C.c_void_p()
    assert lib.mvrl_policy_create_head(C.byref(h), 0, 9, 6, 2) == -1 and b"head" in lib.mvrl_last_error()
    with pytest.raises(RuntimeError):
        SquashedGaussianPolicy(9, 6, device=DEV, action_noise_std=-0.1)
    with pytest.raises(ValueError):
        SquashedGaussianPolicy(9, 6, device=DEV, action_noise_std=[0.1, 0.2])
