"""GPU: ``CriticTarget`` (csrc/mvrl_policy.cu, critic_target_kernel) against a restatement of SB3 SAC / sb3_contrib TQC's
target block in fp64 fed the kernel's own eps - next action, its log-prob, the target critics, the sort / truncation or the
minimum and the affine tail - over shapes, batch sizes and critic configurations; eps against the NumPy Philox restatement
of stream 10; CUDA-graph replays against eager calls; a captured learner step (Polyak update, weight sync, target) with the
new weights on every replay; and the refusals."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from test_critic_target_cpu import stream10_pair

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from marinevehiclereinforcementlearning_b200 import CriticTarget, SquashedGaussianPolicy, _lib
    from marinevehiclereinforcementlearning_b200.policy import critic_param_shapes
    from marinevehiclereinforcementlearning_b200.vec_tools import ReplayBufferSamples
    from test_random_streams_gpu import draw_bound

DEV = "cuda"
SHAPES = [(9, 6), (5, 3), (11, 3), (1, 1), (10, 6)]
SIZES = (1, 127, 128, 129, 4099)
# (kind, n_critics, n_quantiles, drop): n_critics 1 / 2 / 5, n_quantiles 1 / 25 / 32, drop 0 / 2 / n_quantiles - 1
CONFIGS = [("sac", 1, 1, 0), ("sac", 2, 1, 0), ("sac", 5, 1, 0), ("tqc", 2, 25, 2), ("tqc", 1, 1, 0), ("tqc", 5, 32, 31),
           ("tqc", 5, 25, 0), ("tqc", 1, 32, 2), ("tqc", 2, 25, 24)]
# The fp32 actor's bound (test_policy_fp32_gpu.py): |out - fp64| <= TOL * max(1, scale) with scale the batch's largest
# |critic output|; the log-prob (a sum of act_dim terms, each within TOL of its mu / log_std) enters the target times
# gamma * ent_coef.
TOL = 5e-5
GAMMA, ALPHA = 0.99, 0.2


def linear(g, fan_in, fan_out):
    return torch.randn(fan_out, fan_in, generator=g) / math.sqrt(fan_in), torch.rand(fan_out, generator=g) * 0.6 - 0.3


def actor_state_dict(obs_dim, act_dim, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for i, fan_in in zip((0, 2, 4), (obs_dim, 128, 128)):
        sd["latent_pi.%d.weight" % i], sd["latent_pi.%d.bias" % i] = linear(g, fan_in, 128)
    sd["mu.weight"], sd["mu.bias"] = linear(g, 128, act_dim)
    sd["log_std.weight"], sd["log_std.bias"] = linear(g, 128, act_dim)
    sd["log_std.bias"] = torch.rand(act_dim, generator=g) * 1.2 - 1.5
    return sd


def critic_state_dict(obs_dim, act_dim, n_critics, n_out, seed):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for i in range(n_critics):
        for j, fan_in, fan_out in ((0, obs_dim + act_dim, 128), (2, 128, 128), (4, 128, 128), (6, 128, n_out)):
            sd["qf%d.%d.weight" % (i, j)], sd["qf%d.%d.bias" % (i, j)] = linear(g, fan_in, fan_out)
    return sd


def mlp(sd, prefix, x):
    for j in (0, 2, 4):
        x = torch.nn.functional.gelu(x @ sd["%s.%d.weight" % (prefix, j)].to(x).T + sd["%s.%d.bias" % (prefix, j)].to(x))
    return x @ sd["%s.6.weight" % prefix].to(x).T + sd["%s.6.bias" % prefix].to(x)


def restatement(actor_sd, critic_sd, batch, eps, ent_coef, kind, n_critics, drop, gamma=GAMMA):
    """SB3's block in fp64 with the given eps: (target, next_actions, next_log_prob, the batch's largest |critic output|)."""
    x = batch.next_observations.double()
    h = x
    for j in (0, 2, 4):
        h = torch.nn.functional.gelu(h @ actor_sd["latent_pi.%d.weight" % j].to(h).T + actor_sd["latent_pi.%d.bias" % j].to(h))
    mu = h @ actor_sd["mu.weight"].to(h).T + actor_sd["mu.bias"].to(h)
    ls = (h @ actor_sd["log_std.weight"].to(h).T + actor_sd["log_std.bias"].to(h)).clamp(-20.0, 2.0)
    u = mu + ls.exp() * eps.double()
    a = torch.tanh(u)
    logp = torch.distributions.Normal(mu, ls.exp()).log_prob(u).sum(1) - torch.log(1.0 - a * a + 1e-6).sum(1)
    q = torch.stack([mlp(critic_sd, "qf%d" % i, torch.cat([x, a], 1)) for i in range(n_critics)], 1)   # [B, n_critics, n_out]
    if kind == "tqc":
        n_q = q.shape[2]
        qs, _ = torch.sort(q.reshape(q.shape[0], -1))
        qs = qs[:, :n_critics * (n_q - drop)]
    else:
        qs, _ = torch.min(q.reshape(q.shape[0], -1), dim=1, keepdim=True)
    target = batch.rewards.double() + (1 - batch.dones.double()) * gamma * (qs - float(ent_coef) * logp.reshape(-1, 1))
    return target, a, logp, float(q.abs().max())


def make_batch(obs_dim, act_dim, b, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    obs = torch.rand((b, obs_dim), generator=g, device=DEV) * 2 - 1
    rew = torch.rand((b, 1), generator=g, device=DEV) * 2 - 1
    done = (torch.rand((b, 1), generator=g, device=DEV) < 0.3).float()
    return ReplayBufferSamples(torch.zeros((b, obs_dim), device=DEV), torch.zeros((b, act_dim), device=DEV), obs, done, rew)


def make(obs_dim, act_dim, kind, n_critics, n_q, drop, seed=0):
    asd = actor_state_dict(obs_dim, act_dim, seed=obs_dim * 10 + act_dim)
    csd = critic_state_dict(obs_dim, act_dim, n_critics, n_q, seed=seed + 100 * n_critics + n_q)
    actor = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, seed=3, precision="fp32").load_state_dict(asd)
    tgt = CriticTarget(actor, kind=kind, n_critics=n_critics, n_quantiles=n_q, top_quantiles_to_drop_per_net=drop, gamma=GAMMA,
                       seed=seed).load_state_dict(csd)
    return asd, csd, actor, tgt


def run(tgt, batch, ent_coef):
    b = batch.next_observations.shape[0]
    na, eps = (torch.full((b, tgt.act_dim), 7.0, device=DEV) for _ in range(2))
    lp = torch.full((b,), 7.0, device=DEV)
    y = tgt(batch, ent_coef, next_actions=na, next_log_prob=lp, eps=eps)
    torch.cuda.synchronize()
    return y, na, lp, eps


def check(y, na, lp, eps, asd, csd, batch, cfg, worst):
    kind, n_critics, n_q, drop = cfg
    ref, a_ref, lp_ref, qscale = restatement(asd, csd, batch, eps, ALPHA, kind, n_critics, drop)
    act_dim = a_ref.shape[1]
    assert y.shape == ref.shape and bool(torch.isfinite(y).all())
    e_a = float((na.double() - a_ref).abs().max())
    e_lp = float(((lp.double() - lp_ref).abs() / lp_ref.abs().clamp(min=1.0)).max())
    lp_tol = 4 * TOL * act_dim
    e_y = float((y.double() - ref).abs().max()) / (TOL * max(1.0, qscale) + GAMMA * ALPHA * lp_tol * max(1.0, float(lp_ref.abs().max())))
    worst["a"], worst["lp"], worst["y"] = max(worst["a"], e_a), max(worst["lp"], e_lp), max(worst["y"], e_y)
    assert e_a <= TOL and e_lp <= lp_tol and e_y <= 1.0, (cfg, e_a, e_lp, e_y)
    if kind == "tqc":
        assert bool((y[:, 1:] >= y[:, :-1]).all())   # (1 - d) gamma >= 0: the labels keep the ascending order of the values


@pytest.mark.parametrize("cfg", CONFIGS, ids=["%s-%dx%d-drop%d" % c for c in CONFIGS])
@pytest.mark.parametrize("obs_dim,act_dim", SHAPES)
def test_target_matches_fp64_restatement(obs_dim, act_dim, cfg):
    """target, next_actions and next_log_prob against the fp64 restatement fed the kernel's eps, for B = 1 .. 4099 (and
    131 072 for two configurations), dones mixed, ent_coef as a float and as a device tensor."""
    kind, n_critics, n_q, drop = cfg
    asd, csd, actor, tgt = make(obs_dim, act_dim, *cfg)
    sizes = SIZES + ((131072,) if (obs_dim, act_dim) == (9, 6) and cfg in (CONFIGS[3], CONFIGS[1]) else ())
    worst = {"a": 0.0, "lp": 0.0, "y": 0.0}
    for i, b in enumerate(sizes):
        batch = make_batch(obs_dim, act_dim, b, seed=b)
        alpha = ALPHA if i % 2 == 0 else torch.tensor([ALPHA], device=DEV)
        y, na, lp, eps = run(tgt, batch, alpha)
        assert y.shape == (b, n_critics * (n_q - drop) if kind == "tqc" else 1)
        check(y, na, lp, eps, asd, csd, batch, cfg, worst)
    assert int(tgt.calls[0]) == len(sizes) and int(tgt.calls[1]) == 0
    print("critic target %s (%d, %d): max |a - fp64| %.3g, rel |logp - fp64| %.3g, |target - fp64| / bound %.3g"
          % (cfg, obs_dim, act_dim, worst["a"], worst["lp"], worst["y"]))


def test_float_and_tensor_ent_coef_agree_and_dones_cut_the_bootstrap():
    """The same call number gives the same bits with ent_coef as a float and as a tensor; rows with done = 1 are the reward."""
    asd, csd, actor, tgt = make(9, 6, "tqc", 2, 25, 2)
    batch = make_batch(9, 6, 1000, seed=4)
    y1 = run(tgt, batch, 0.3)[0]
    tgt.calls.zero_()
    y2 = run(tgt, batch, torch.tensor([0.3], device=DEV))[0]
    assert torch.equal(y1, y2)
    d = batch.dones.squeeze(1) == 1
    assert bool(d.any()) and torch.equal(y1[d], batch.rewards[d].expand(-1, y1.shape[1]))


def test_eps_matches_numpy_philox_stream_10():
    """Every eps entry of 4099 rows at call numbers 0, 1 and 2^32 + 3 within the bound of its draw against the NumPy
    restatement (test_random_streams_gpu.draw_bound); another call number draws different values."""
    asd, csd, actor, tgt = make(10, 6, "tqc", 2, 25, 2, seed=0)
    tgt.seed = 0xD1B54A32D192ED03
    b = 4099
    batch = make_batch(10, 6, b, seed=1)
    worst = 0.0
    prev = None
    for call in (0, 1, 2 ** 32 + 3):
        tgt.calls.copy_(torch.tensor([call, 0]))
        eps = run(tgt, batch, ALPHA)[3].cpu().numpy().astype(np.float64)
        for pr in range(3):
            k1, k2, z0, z1 = stream10_pair(tgt.seed, np.arange(b), call, pr)
            for c, z in enumerate((z0, z1)):
                d = np.abs(eps[:, 2 * pr + c] - z)
                bound = draw_bound(k1, k2, z)
                assert np.all(d <= bound), (call, pr, c, float((d / bound).max()))
                worst = max(worst, float((d / bound).max()))
        if prev is not None:
            assert np.mean(prev == eps) < 0.01
        prev = eps
        assert int(tgt.calls[0]) == call + 1
    print("stream 10 eps: worst |kernel - numpy| / bound %.3f" % worst)


def test_graph_replays_equal_eager_calls():
    """T = 3 calls captured in one CUDA graph and replayed R = 4 times give the bits of 12 eager calls; calls advances by 12."""
    asd, csd, actor, tgt = make(11, 3, "tqc", 5, 25, 2)
    batches = [make_batch(11, 3, b, seed=b) for b in (300, 129, 1)]
    alpha = torch.tensor([ALPHA], device=DEV)
    T, R = len(batches), 4
    tgt.calls.zero_()
    eager = []
    for _ in range(R):
        for batch in batches:
            eager.append(tgt(batch, alpha))
    torch.cuda.synchronize()
    assert int(tgt.calls[0]) == T * R
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for batch in batches:
            tgt(batch, alpha)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    tgt.calls.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        outs = [tgt(batch, alpha) for batch in batches]
    assert int(tgt.calls[0]) == 0
    replayed = []
    for _ in range(R):
        g.replay()
        replayed += [o.clone() for o in outs]
    torch.cuda.synchronize()
    assert int(tgt.calls[0]) == T * R and int(tgt.calls[1]) == 0
    for e, r in zip(eager, replayed):
        assert torch.equal(e, r)
    assert not torch.equal(replayed[0], replayed[T])


def test_captured_learner_step_uses_the_new_weights():
    """A graph of: Polyak update of the target critics (torch._foreach_lerp_), an in-place actor update, tgt.sync_weights(),
    actor_t.sync_weights() and tgt(batch, ent_coef) - on every replay the target equals the restatement with the weights
    of that replay."""
    obs_dim, act_dim, cfg = 9, 6, ("tqc", 2, 25, 2)
    asd = {k: v.to(DEV) for k, v in actor_state_dict(obs_dim, act_dim, 5).items()}
    online = {k: v.to(DEV) for k, v in critic_state_dict(obs_dim, act_dim, 2, 25, 6).items()}
    target = {k: v.to(DEV) for k, v in critic_state_dict(obs_dim, act_dim, 2, 25, 7).items()}
    actor = SquashedGaussianPolicy(obs_dim, act_dim, device=DEV, precision="fp32").load_state_dict(asd, share=True)
    tgt = CriticTarget(actor, n_critics=2, n_quantiles=25, top_quantiles_to_drop_per_net=2, gamma=GAMMA).load_state_dict(
        {"critic." + k: v for k, v in online.items()} | {"critic_target." + k: v for k, v in target.items()}, share=True)
    assert all(tgt.params[k].data_ptr() == target[k].data_ptr() for k in target)
    batch = make_batch(obs_dim, act_dim, 777, seed=3)
    alpha = torch.tensor([ALPHA], device=DEV)
    eps = torch.empty((777, act_dim), device=DEV)
    keys = list(critic_param_shapes(obs_dim, act_dim, 2, 25))
    delta = {k: torch.randn(v.shape, generator=torch.Generator().manual_seed(1)).to(DEV) * 1e-2 for k, v in asd.items()}

    def step():
        torch._foreach_lerp_([target[k] for k in keys], [online[k] for k in keys], 0.05)
        for k in asd:
            asd[k].add_(delta[k])
        tgt.sync_weights()
        actor.sync_weights()
        return tgt(batch, alpha, eps=eps)

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        y = step()
    worst = 0.0
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        ref, _, lp_ref, qscale = restatement(asd, target, batch, eps, ALPHA, "tqc", 2, 2)
        bound = TOL * max(1.0, qscale) + GAMMA * ALPHA * 4 * TOL * act_dim * max(1.0, float(lp_ref.abs().max()))
        e = float((y.double() - ref).abs().max()) / bound
        worst = max(worst, e)
        assert e <= 1.0, e
    print("captured learner step: |target - fp64 with the replay's weights| / bound %.3g" % worst)


def test_refusals():
    asd, csd, actor, tgt = make(9, 6, "tqc", 2, 25, 2)
    batch = make_batch(9, 6, 64, seed=0)
    cpu = ReplayBufferSamples(*[t.cpu() for t in batch])
    f64 = ReplayBufferSamples(*[t.double() for t in batch])
    for bad in (cpu, f64):
        with pytest.raises(ValueError):
            tgt(bad, ALPHA)
    for alpha in (torch.tensor([0.1, 0.2], device=DEV), torch.tensor([0.1]), torch.tensor([0.1], dtype=torch.float64, device=DEV)):
        with pytest.raises(ValueError, match="ent_coef"):
            tgt(batch, alpha)
    with pytest.raises(ValueError, match="next_actions"):
        tgt(batch, ALPHA, next_actions=torch.empty((64, 5), device=DEV))
    with pytest.raises(ValueError, match="fp32"):
        CriticTarget(SquashedGaussianPolicy(9, 6, device=DEV))
    with pytest.raises(ValueError, match="share=True"):
        tgt.load_state_dict(csd, share=True)   # CPU tensors
    with pytest.raises(ValueError):
        CriticTarget(actor, n_critics=3).load_state_dict(csd)
    # the C entry: host memory, an actor with other dims, a drop that keeps nothing
    lib = _lib.load()
    out = torch.empty((64, 46), device=DEV)
    alpha = torch.tensor([ALPHA], device=DEV)
    st = _lib.current_stream(tgt.device)

    def call(actor_h, obs, drop=2):
        return lib.mvrl_critic_target(tgt._h, actor_h, 64, _lib.ptr(obs), _lib.ptr(batch.rewards), _lib.ptr(batch.dones), _lib.ptr(alpha),
                                      GAMMA, drop, 0, _lib.ptr(tgt.calls), _lib.ptr(out), None, None, None, st)
    assert call(actor._h, batch.next_observations.cpu()) == -1 and b"not device memory" in lib.mvrl_last_error()
    other = SquashedGaussianPolicy(9, 5, device=DEV, precision="fp32")
    assert call(other._h, batch.next_observations) == -1 and b"actor" in lib.mvrl_last_error()
    assert call(actor._h, batch.next_observations, drop=25) == -1 and b"drop_per_net" in lib.mvrl_last_error()
    h = C.c_void_p()
    assert lib.mvrl_critic_create(C.byref(h), 0, 9, 6, 0, 2, 25) == -1 and b"n_quantiles" in lib.mvrl_last_error()
    assert lib.mvrl_critic_create(C.byref(h), 0, 9, 6, 1, 6, 25) == -1 and b"n_critics" in lib.mvrl_last_error()
    assert call(actor._h, batch.next_observations) == 0
    torch.cuda.synchronize()
