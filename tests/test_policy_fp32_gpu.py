"""GPU: the fp32 precision of the fused rollout actor (csrc/mvrl_policy.cu, policy_act_fp32_kernel) - both heads against the
network evaluated in fp64 with the erf GELU, and SB3's predict against the same network in fp32 on the CPU; the noise
against the bf16 precision's, bit for bit."""
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
SHAPES = [(9, 6), (5, 3), (11, 3), (1, 1), (16, 8)]
SIZES = (1, 37, 127, 129, 5000, 131072)
# Observations in [-1, 1]: |out - out_fp64| <= TOL * max(1, |out_fp64|) element by element.  A CPU model of the split
# (bf16 hi / lo operands, exact products, fp32 accumulation per K = 16 step) gives 7e-6 .. 8e-6; the margin covers the
# tensor core's own accumulation order.  Single-pass bf16 is ~4e-3 in the same model.
# Observations in [-30, 30]: the split keeps 16 significant bits of every operand, so the error follows the size of the
# terms summed, not of the result - an output near 0 built from hidden activations of ~30 carries their absolute error.
# There the bound is TOL * max(1, the batch's largest |head-layer output|) (the model: 3.3e-4 where |mu| reaches 30,
# 1.1e-5 of that scale); for the fixed head the scale is that of its pre-tanh output (tanh has slope <= 1).
TOL = 5e-5
MIN_GAIN = 20.0   # the fp32 handle's worst error is at least this many times below the bf16 handle's on the same inputs


def random_network(obs_dim, act_dim, seed, log_std_bias=(-1.5, -0.3)):
    """Hidden layers [(W, b)] * 3 and head layers [(W, b)] (mu, log_std), fp32 CPU, nn.Linear layout, non-zero biases."""
    g = torch.Generator().manual_seed(seed)

    def linear(fan_in, fan_out):
        return torch.randn(fan_out, fan_in, generator=g) / math.sqrt(fan_in), torch.rand(fan_out, generator=g) * 0.6 - 0.3
    hidden = [linear(obs_dim, 128), linear(128, 128), linear(128, 128)]
    mu, ls = linear(128, act_dim), linear(128, act_dim)
    lo, hi = log_std_bias
    ls = (ls[0], torch.rand(act_dim, generator=g) * (hi - lo) + lo)
    return hidden, [mu, ls]


def forward(hidden, heads, obs_nk, dtype):
    """The network with torch.nn.GELU() (erf form) in `dtype` on obs_nk's device: the head layers' outputs [N, act_dim]."""
    h = obs_nk.to(dtype)
    for W, b in hidden:
        h = torch.nn.functional.gelu(h @ W.to(h).T + b.to(h))
    return [h @ W.to(h).T + b.to(h) for W, b in heads]


def fixed_policy(obs_dim, act_dim, hidden, head, precision, seed=3):
    pol = MlpGaussianPolicy(obs_dim, act_dim, device=DEV, seed=seed, precision=precision)
    pol.weights = [W for W, _ in hidden] + [head[0]]
    pol.biases = [b for _, b in hidden] + [head[1]]
    pol.log_std = torch.linspace(-1.2, -0.2, act_dim)
    pol.sync_weights()
    return pol


def squashed_state_dict(hidden, heads):
    sd = {}
    for i, (W, b) in zip((0, 2, 4), hidden):
        sd["latent_pi.%d.weight" % i], sd["latent_pi.%d.bias" % i] = W, b
    (sd["mu.weight"], sd["mu.bias"]), (sd["log_std.weight"], sd["log_std.bias"]) = heads
    return sd


def squashed_policy(obs_dim, act_dim, sd, precision, noise=None, seed=3):
    return SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, seed=seed, action_noise_std=noise, precision=precision).load_state_dict(sd)


def buffers(obs_dim, act_dim, n, seed=0, scale=1.0):
    ld = (n + 31) // 32 * 32
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.zeros((obs_dim, ld), device=DEV)
    obs[:, :n] = (torch.rand((obs_dim, n), generator=g, device=DEV) * 2 - 1) * scale
    z = lambda k: torch.full((k, ld), 7.0, device=DEV)
    return dict(obs=obs, act=z(act_dim), mean=z(act_dim), log_std=z(act_dim), eps=z(act_dim), logp=torch.full((ld,), 7.0, device=DEV))


def run(pol, b, n, env_id0=11, step=4, deterministic=False):
    squashed = isinstance(pol, SquashedGaussianPolicy)
    pol.act_into(b["obs"], b["act"], n, logp=b["logp"], mean=b["mean"], eps=b["eps"], log_std=b["log_std"] if squashed else None,
                 env_id0=env_id0, step=step, deterministic=deterministic)
    torch.cuda.synchronize()
    return b


def rel_err(out, ref, scale=None):
    """max |out - ref| / max(1, |ref|) element by element, or / max(1, scale) when a batch scale is given."""
    d = (out.double() - ref).abs()
    return float((d / ref.abs().clamp(min=1.0)).max()) if scale is None else float(d.max()) / max(1.0, scale)


def cases():
    """(n, observation scale): every size with observations in [-1, 1], and one batch with observations in [-30, 30]."""
    return [(n, 1.0) for n in SIZES] + [(5000, 30.0)]


def check_untouched(b, n, keys):
    for k in keys:
        assert bool((b[k][:, n:] == 7.0).all()), k
    assert bool((b["logp"][n:] == 7.0).all())


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_squashed_fp32_matches_fp64_network(obs_dim, act_dim):
    """mu and the clamped log_std of the fp32 squashed head against the fp64 network, with log_std biases on both sides of
    the clamp; act and logp by SB3's formulas (fp64) from the kernel's own mu / log_std / eps; nothing written at or beyond
    row n; the bf16 handle's error on the same inputs is at least MIN_GAIN times larger."""
    hidden, heads = random_network(obs_dim, act_dim, seed=obs_dim * 10 + act_dim, log_std_bias=(-21.0, 2.5))
    sd = squashed_state_dict(hidden, heads)
    pols = {p: squashed_policy(obs_dim, act_dim, sd, p) for p in ("fp32", "bf16")}
    worst = {"fp32": 0.0, "bf16": 0.0, "act": 0.0, "logp": 0.0, "cpu32": 0.0}
    for n, scale in cases():
        out = {p: run(pol, buffers(obs_dim, act_dim, n, scale=scale), n) for p, pol in pols.items()}
        x = out["fp32"]["obs"][:, :n].T
        mu64, ls64 = forward(hidden, heads, x, torch.float64)
        ls64 = ls64.clamp(-20.0, 2.0)
        bscale = None if scale == 1.0 else float(max(mu64.abs().max(), ls64.abs().max()))
        for p, b in out.items():
            e = max(rel_err(b["mean"][:, :n].T, mu64, bscale), rel_err(b["log_std"][:, :n].T, ls64, bscale))
            worst[p] = max(worst[p], e)
            if p == "fp32" and bscale is not None:
                worst["x30_abs"] = float(max((b["mean"][:, :n].T - mu64).abs().max(), (b["log_std"][:, :n].T - ls64).abs().max()))
                worst["x30_scale"] = bscale
        b = out["fp32"]
        mu, ls, eps, act, logp = b["mean"][:, :n].T, b["log_std"][:, :n].T, b["eps"][:, :n].T, b["act"][:, :n].T, b["logp"][:n]
        e_mu, e_ls = rel_err(mu, mu64, bscale), rel_err(ls, ls64, bscale)
        assert e_mu <= TOL and e_ls <= TOL, (n, scale, e_mu, e_ls)
        if n <= 5000:   # SB3's own arithmetic: the same network in fp32 on the CPU
            mu32, ls32 = forward(hidden, heads, x.cpu(), torch.float32)
            worst["cpu32"] = max(worst["cpu32"], rel_err(mu.cpu(), mu32.double(), bscale), rel_err(ls.cpu(), ls32.clamp(-20.0, 2.0).double(), bscale))
        m, s, e_, a_ = (t.double() for t in (mu, ls, eps, act))
        std = s.exp()
        u = m + std * e_
        lp_ref = torch.distributions.Normal(m, std).log_prob(u).sum(1) - torch.log(1.0 - a_ * a_ + 1e-6).sum(1)
        e_act, e_lp = float((a_ - torch.tanh(u)).abs().max()), float((logp.double() - lp_ref).abs().max())
        assert e_act < 2e-6 and e_lp < 1e-5 * act_dim, (n, e_act, e_lp)
        assert bool((act.abs() <= 1.0).all())
        check_untouched(b, n, ("act", "mean", "log_std", "eps"))
        worst["act"], worst["logp"] = max(worst["act"], e_act), max(worst["logp"], e_lp)
    print("fp32 squashed head (%d, %d): max rel |mu, log_std - fp64| %.3g (bf16 handle %.3g, x%.0f); - fp32 CPU %.3g; "
          "obs x30: abs %.3g at scale %.3g; |act - formula| %.3g; |logp - formula| %.3g"
          % (obs_dim, act_dim, worst["fp32"], worst["bf16"], worst["bf16"] / max(worst["fp32"], 1e-30), worst["cpu32"], worst["x30_abs"],
             worst["x30_scale"], worst["act"], worst["logp"]))
    assert worst["bf16"] >= MIN_GAIN * worst["fp32"], worst


@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_fixed_fp32_matches_fp64_network(obs_dim, act_dim):
    """The fp32 fixed head: its mean tanh(W4 h + b4) against the fp64 network; act = clip(mean + std eps, -1, 1) and
    logp = -sum eps^2 / 2 - sum log_std from the kernel's own mean / eps; nothing written at or beyond row n; the bf16
    handle's error on the same inputs is at least MIN_GAIN times larger."""
    hidden, heads = random_network(obs_dim, act_dim, seed=obs_dim * 10 + act_dim + 1)
    pols = {p: fixed_policy(obs_dim, act_dim, hidden, heads[0], p) for p in ("fp32", "bf16")}
    worst = {"fp32": 0.0, "bf16": 0.0, "act": 0.0, "logp": 0.0}
    std = pols["fp32"].log_std.double().exp().to(DEV)
    for n, scale in cases():
        out = {p: run(pol, buffers(obs_dim, act_dim, n, scale=scale), n) for p, pol in pols.items()}
        x = out["fp32"]["obs"][:, :n].T
        pre64 = forward(hidden, heads[:1], x, torch.float64)[0]
        mean64 = torch.tanh(pre64)
        bscale = None if scale == 1.0 else float(pre64.abs().max())
        for p, b in out.items():
            worst[p] = max(worst[p], rel_err(b["mean"][:, :n].T, mean64, bscale))
            if p == "fp32" and bscale is not None:
                worst["x30_abs"], worst["x30_scale"] = float((b["mean"][:, :n].T - mean64).abs().max()), bscale
        b = out["fp32"]
        mean, eps, act, logp = b["mean"][:, :n].T, b["eps"][:, :n].T, b["act"][:, :n].T, b["logp"][:n]
        assert rel_err(mean, mean64, bscale) <= TOL, (n, scale, rel_err(mean, mean64, bscale))
        a_ref = (mean.double() + std * eps.double()).clamp(-1.0, 1.0)
        lp_ref = -0.5 * (eps.double() ** 2).sum(1) - float(pols["fp32"].log_std.double().sum())
        e_act, e_lp = float((act.double() - a_ref).abs().max()), float((logp.double() - lp_ref).abs().max())
        assert e_act < 2e-6 and e_lp < 1e-5 * act_dim, (n, e_act, e_lp)
        check_untouched(b, n, ("act", "mean", "eps"))
        worst["act"], worst["logp"] = max(worst["act"], e_act), max(worst["logp"], e_lp)
    print("fp32 fixed head (%d, %d): max rel |tanh mean - fp64| %.3g (bf16 handle %.3g, x%.0f); obs x30: abs %.3g at pre-tanh scale %.3g; "
          "|act - formula| %.3g; |logp - formula| %.3g"
          % (obs_dim, act_dim, worst["fp32"], worst["bf16"], worst["bf16"] / max(worst["fp32"], 1e-30), worst["x30_abs"], worst["x30_scale"],
             worst["act"], worst["logp"]))
    assert worst["bf16"] >= MIN_GAIN * worst["fp32"], worst


def test_fixed_fp32_mean_is_the_accurate_tanh():
    """With zero head weights the fixed head's mean is tanh(b4) of an exact fp32 b4: within 3e-7 (the accurate tanhf, a
    couple of ulp) of tanh in fp64, over 64 values in [-3, 3].  tanh.approx is ~2^-11 relative."""
    hidden, heads = random_network(9, 8, seed=6)
    pol = fixed_policy(9, 8, hidden, (torch.zeros(8, 128), torch.zeros(8)), "fp32")
    b4s = torch.linspace(-3.0, 3.0, 64).reshape(8, 8)
    worst = 0.0
    for b4 in b4s:
        pol.biases[3] = b4.clone()
        pol.sync_weights()
        b = run(pol, buffers(9, 8, 200), 200, deterministic=True)
        ref = torch.tanh(b4.double()).to(DEV)[:, None]
        worst = max(worst, float((b["mean"][:, :200].double() - ref).abs().max()))
        assert torch.equal(b["act"][:, :200], b["mean"][:, :200])
    print("fp32 fixed head: max |tanh(b4) - fp64| %.3g" % worst)
    assert worst < 3e-7, worst


def test_trained_tqc_actor_predict_matches_sb3():
    """A whole TQC policy state dict (actor.* and critic.* keys): predict(obs, deterministic=True) of the fp32 policy is
    tanh(mu) of the network in fp32 on the CPU (SB3's predict) within TOL."""
    hidden, heads = random_network(9, 6, seed=8)
    actor = squashed_state_dict(hidden, heads)
    g = torch.Generator().manual_seed(1)
    sd = {"actor." + k: v for k, v in actor.items()}
    sd.update({"critic.qf0.0.weight": torch.randn(128, 15, generator=g), "critic.qf0.0.bias": torch.zeros(128),
               "critic_target.qf0.0.weight": torch.randn(128, 15, generator=g)})
    pol = SquashedGaussianPolicy(9, 6, device=DEV, action_noise_std=0.5, precision="fp32").load_state_dict(sd)
    assert pol.precision == "fp32"
    obs = np.random.default_rng(0).uniform(-1, 1, (300, 9)).astype(np.float32)
    a, _ = pol.predict(obs, deterministic=True)
    mu32, _ = forward(hidden, heads, torch.as_tensor(obs), torch.float32)
    err = float(np.abs(a - torch.tanh(mu32).numpy()).max())
    print("fp32 predict: max |predict - tanh(mu) of the fp32 CPU network| %.3g" % err)
    assert a.shape == (300, 6) and err < TOL
    a1, _ = pol.predict(obs[0], deterministic=True)
    assert a1.shape == (6,) and np.array_equal(a1, a[0])


@pytest.mark.parametrize("obs_dim,act_dim", [(9, 6), (16, 8), (1, 1)])
def test_same_randomness_as_bf16(obs_dim, act_dim):
    """Same seed, env_id0 and step: eps bitwise equal between a bf16 and an fp32 handle (both heads); with zero head
    weights (mu = b_mu and log_std = b_log_std exactly in both) the squashed act with action noise and logp are bitwise
    equal too; two shards with env_id0 offsets give the bits of one launch."""
    hidden, heads = random_network(obs_dim, act_dim, seed=5)
    zero = [(torch.zeros_like(W), b) for W, b in heads]
    sd0 = squashed_state_dict(hidden, zero)
    n = 1000
    sq = {p: squashed_policy(obs_dim, act_dim, sd0, p, noise=0.3) for p in ("bf16", "fp32")}
    fx = {p: fixed_policy(obs_dim, act_dim, hidden, heads[0], p) for p in ("bf16", "fp32")}
    for pols in (sq, fx):
        out = {p: run(pol, buffers(obs_dim, act_dim, n, seed=2), n, env_id0=5, step=9) for p, pol in pols.items()}
        assert torch.equal(out["bf16"]["eps"], out["fp32"]["eps"])
        assert bool((out["fp32"]["eps"][:, :n] != 0.0).any())
    zs = {p: run(pol, buffers(obs_dim, act_dim, n, seed=2), n, env_id0=5, step=9) for p, pol in sq.items()}
    for k in ("mean", "log_std", "act", "logp"):
        assert torch.equal(zs["bf16"][k], zs["fp32"][k]), k
    # sharding, with a network in front of the head
    pol = squashed_policy(obs_dim, act_dim, squashed_state_dict(hidden, heads), "fp32", noise=0.3)
    lo = 512
    b = run(pol, buffers(obs_dim, act_dim, n, seed=2), n, env_id0=0, step=7)
    obs2 = b["obs"][:, lo:lo + 512].contiguous()
    act2, eps2, mean2 = (torch.zeros((act_dim, 512), device=DEV) for _ in range(3))
    pol.act_into(obs2, act2, n - lo, eps=eps2, mean=mean2, env_id0=lo, step=7)
    torch.cuda.synchronize()
    assert torch.equal(eps2[:, :n - lo], b["eps"][:, lo:n])
    assert torch.equal(mean2[:, :n - lo], b["mean"][:, lo:n])
    assert torch.equal(act2[:, :n - lo], b["act"][:, lo:n])


def test_log_std_clamp():
    """log_std biases of +-30 give exactly 2 / -20 in the fp32 squashed head, with finite act and logp."""
    hidden, heads = random_network(9, 6, seed=4)
    for bias, want in ((30.0, 2.0), (-30.0, -20.0)):
        sd = squashed_state_dict(hidden, heads)
        sd["log_std.bias"] = torch.full((6,), bias)
        pol = squashed_policy(9, 6, sd, "fp32")
        n = 1000
        b = run(pol, buffers(9, 6, n), n)
        assert bool((b["log_std"][:, :n] == want).all())
        assert bool(torch.isfinite(b["act"][:, :n]).all()) and bool(torch.isfinite(b["logp"][:n]).all())


@pytest.mark.parametrize("which", ["rov6", "rov3", "auv"])
def test_closed_loop(which):
    """20 steps of pol.act(env); env.step() with an fp32 squashed policy on the env's own buffers: state and logp finite,
    |act| <= 1."""
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
    pol = SquashedGaussianPolicy(env.lenObs, env.lenAction, device=DEV, seed=1, action_noise_std=0.1, precision="fp32")
    env.reset()
    logp = torch.empty(env.ld, device=DEV)
    for _ in range(20):
        pol.act(env, logp=logp)
        assert float(env.actions_fm.abs().max()) <= 1.0
        env.step()
        assert bool(torch.isfinite(logp[:n]).all())
    assert bool(torch.isfinite(env.state if which == "auv" else env.systemState).all())


def test_rejections(monkeypatch):
    """MVRL_EINVAL for an unknown precision (naming it) and for an fp32 handle with MVRL_POLICY_MMA_SYNC=1 (naming the
    variable); the bf16 handle is still created with it; an unknown precision string is a ValueError."""
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, 1, 2) == -1 and b"precision" in lib.mvrl_last_error()
    monkeypatch.setenv("MVRL_POLICY_MMA_SYNC", "1")
    for head in (0, 1):
        assert lib.mvrl_policy_create_ex(C.byref(h), 0, 9, 6, head, 1) == -1 and b"MVRL_POLICY_MMA_SYNC" in lib.mvrl_last_error()
    with pytest.raises(RuntimeError, match="MVRL_POLICY_MMA_SYNC"):
        SquashedGaussianPolicy(9, 6, device=DEV, precision="fp32")
    assert SquashedGaussianPolicy(9, 6, device=DEV).precision == "bf16"
    with pytest.raises(ValueError):
        MlpGaussianPolicy(9, 6, device=DEV, precision="fp16")
